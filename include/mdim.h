/*
 * mdim.h — C ABI of the B200-native View→collect() hot path of apt1002/multidimension.
 *
 * What this boundary replaces.  The reference has no FFI: `collect()` is a provided method of
 * the `View` trait (reference src/view.rs:146-150) that drives `View::each` (src/view.rs:250-252)
 * into the sink plugin `NewView::new_view` (src/view.rs:20-38, impl for Array src/array.rs:103-114)
 * one `Push::push` at a time (src/view.rs:8-11, src/array.rs:99-101).  That element-at-a-time
 * protocol is host-serial, so a device path needs a whole-expression entry point: the host side
 * (Rust `DeviceArray`, the C++ mirror in include/mdim/view.hpp, or the Python mirror in
 * multidimension_b200/) lowers the lazy View tree into the flattened, position-space descriptor
 * below (`mdim_expr`) and calls `mdim_collect`, which runs the whole chain as ONE fused pass of a
 * hand-written sm_100a kernel.  INTEGRATION.md shows the Rust binding a maintainer would add.
 *
 * Position space.  Every reference index type flattens (src/tuple.rs:60-176) to an ordered list
 * of leaf axes; `Index::to_usize` (src/index.rs:75-154) is row-major over that list and
 * `Index::each` visits it last-axis-fastest.  The descriptor therefore carries only the run-time
 * leaf lengths of the OUTPUT index (plus optional trailing reduction axes) and, per node, strides
 * against those iteration axes.  `Iso`/`Coat`/`Transpose`/`Row`/`Column`/broadcast all disappear
 * into strides and offsets at lowering time.
 *
 * Plain pointers and sizes only; no C++/torch types.  All functions return an mdim_status.
 * A context is single-threaded (the caller serialises), one context per GPU per process.
 * There is NO CPU fallback: every entry point that computes fails with MDIM_ERR_CUDA when no
 * sm_100 device is usable.
 */
#ifndef MDIM_H
#define MDIM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDIM_ABI_VERSION 1
#define MDIM_MAX_RANK 8   /* output leaf axes + reduction leaf axes */
#define MDIM_MAX_NODES 48 /* nodes in one fused expression */
#define MDIM_MAX_PEERS 8  /* shards of a peer-mapped gather source (one 8-GPU NVSwitch box) */
#define MDIM_MAX_OUTS 4   /* scalar leaves of a tuple-typed element collected in ONE launch (MDIM_NODE_TUPLE) */

/* Layout of tuple-typed Arrays.  Rust leaves the layout of (T, U) unspecified (no repr(C) on tuples), so the device
 * declares its own: an Array whose element type is a tuple is a STRUCTURE OF ARRAYS — one dense row-major run per
 * scalar leaf of the (flattened) element type, in flattening order, each exactly as a scalar-typed Array of that leaf
 * type would be stored.  `Array<I, (usize, f32)>` is a u64 run of I::length elements and an f32 run of the same length;
 * element k of the Array is (run0[k], run1[k]).  mdim_collect_tuple fills all runs from ONE kernel launch (shared operands
 * are read once); a host `Vec<(T, U)>` is obtained by interleaving the downloaded runs (DeviceArray::to_raw). */

/* ---- status codes: every reference panic site maps to one of these (SURVEY.md §8b) ---------- */
typedef enum mdim_status {
    MDIM_OK = 0,
    MDIM_ERR_OOB = 1,         /* src/int.rs:17  "Index {:?} is out of bounds for size {:?}"         */
    MDIM_ERR_SIZE = 2,        /* src/array.rs:12 length mismatch; src/broadcast.rs:38 "Unequal sizes" */
    MDIM_ERR_UNSUPPORTED = 3, /* expression is valid in the reference but not lowerable to a device  */
    MDIM_ERR_CUDA = 4,        /* CUDA runtime/driver failure, or no sm_100 device                    */
    MDIM_ERR_ARITH = 5,       /* integer division/remainder by zero, or MIN / -1 (Rust panics)       */
    MDIM_ERR_INVALID = 6,     /* malformed descriptor (bad arity, dtype mismatch, null pointer ...)   */
    MDIM_ERR_NOMEM = 7,
    MDIM_ERR_NCCL = 8         /* NCCL missing or a collective failed (multi-GPU entry points only)             */
} mdim_status;

/* ---- element types. `usize` of the reference is MDIM_U64 ------------------------------------- */
typedef enum mdim_dtype {
    MDIM_U8 = 0, /* also Rust bool (0/1) */
    MDIM_I32 = 1,
    MDIM_U32 = 2,
    MDIM_I64 = 3,
    MDIM_U64 = 4,
    MDIM_F32 = 5,
    MDIM_F64 = 6,
    MDIM_DTYPE_COUNT = 7
} mdim_dtype;

/* ---- binary operator vocabulary = the reference's uninstantiable enums, src/ops.rs:23-129 ---- */
typedef enum mdim_binary_op {
    MDIM_ADD = 0, /* ops::Add    src/ops.rs:33  */
    MDIM_SUB = 1, /* ops::Sub    src/ops.rs:43  */
    MDIM_MUL = 2, /* ops::Mul    src/ops.rs:53  */
    MDIM_DIV = 3, /* ops::Div    src/ops.rs:63  */
    MDIM_REM = 4, /* ops::Rem    src/ops.rs:73  */
    MDIM_AND = 5, /* ops::BitAnd src/ops.rs:83  */
    MDIM_OR = 6,  /* ops::BitOr  src/ops.rs:93  */
    MDIM_XOR = 7, /* ops::BitXor src/ops.rs:103 */
    MDIM_SHL = 8, /* ops::Shl    src/ops.rs:113 */
    MDIM_SHR = 9, /* ops::Shr    src/ops.rs:123 */
    MDIM_BINARY_COUNT = 10
} mdim_binary_op;
/* extra reduction operators accepted by mdim_allreduce only (a fold with a closure `|s, x| s.min(x)`) */
#define MDIM_REDUCE_MIN 100
#define MDIM_REDUCE_MAX 101

/* ---- closed unary vocabulary standing in for `Map`'s opaque closure (src/view.rs:880-889);
 *      same type-level style as ops.rs.  Affine maps such as x*y+1 are spelled with BINARY nodes
 *      and CONST (`Scalar`, src/view.rs:1399-1408) operands, exactly as `a*b + Scalar(1.0)`. ----- */
typedef enum mdim_unary_op {
    MDIM_NEG = 0,  /* std::ops::Neg; wrapping for integers */
    MDIM_NOT = 1,  /* std::ops::Not on integers: bitwise (U8 included).  `!bool` is lowered by the host as x ^ 1 */
    MDIM_ABS = 2,
    MDIM_SQRT = 3, /* f32/f64 only, IEEE correctly rounded */
    MDIM_CAST = 4, /* Rust `as` between the dtypes above; source dtype in mdim_node.src_dtype */
    MDIM_UNARY_COUNT = 5
} mdim_unary_op;

typedef enum mdim_node_kind {
    MDIM_NODE_LEAF = 0,   /* Array as a View: src/array.rs:73-92                                   */
    MDIM_NODE_IOTA = 1,   /* All<I>: src/index.rs:177-186 (value = coordinate, linear combination)  */
    MDIM_NODE_CONST = 2,  /* Scalar<T>: src/view.rs:1399-1408                                       */
    MDIM_NODE_UNARY = 3,  /* Map<V,F> for the closed op set: src/view.rs:880-889                    */
    MDIM_NODE_BINARY = 4, /* Zip<V,W,B>: src/view.rs:1178-1198 (+ Broadcast as zero strides)        */
    MDIM_NODE_DIAG = 5,   /* Diagonal<V>: src/view.rs:846-857                                       */
    MDIM_NODE_GATHER = 6, /* Compose<V,W>: src/view.rs:897-912; MapAxis: src/view.rs:1140-1170      */
    MDIM_NODE_FOLD = 7,   /* rows().map(|r| fold r.each(..)): src/view.rs:617-622,1330-1342,250-252 */
    MDIM_NODE_CONCAT = 8, /* Concat<V,W,I,J>: src/view.rs:920-946 (coord[axis_a[0]] < axis_c[0] ? V : W)  */
    MDIM_NODE_TUPLE = 9,  /* ROOT ONLY: a tuple-typed element — `zip` without an operator (ops::Pair, src/ops.rs:25-29), `enumerate`
                             (src/view.rs:829-838), a compound All<I> (src/index.rs:177-186).  n_comp children (<= MDIM_MAX_OUTS),
                             one per scalar leaf of the element type in flattening order; see "layout of tuple-typed Arrays" */
    MDIM_NODE_KIND_COUNT = 10
} mdim_node_kind;

typedef union mdim_scalar {
    uint64_t u64;
    int64_t i64;
    double f64;
    float f32;
    uint32_t u32;
    int32_t i32;
    uint8_t u8;
} mdim_scalar;

/*
 * One node of the expression, nodes are stored in POST-ORDER (children before parent, left to
 * right), so the array is also a stack program.  Arity: LEAF/IOTA/CONST 0, UNARY 1, BINARY 2,
 * DIAG 1, GATHER n_comp, FOLD 1 (2 when n_comp == 2: the FIRST child is then the initial value, any value tree over
 * the output axes — `let mut s = init.at(i)` — and `imm` is unused), CONCAT 2.  The last node is the root and its dtype is the output dtype.
 *
 * Iteration axes: 0..rank-1 are the output leaf axes, rank..rank+red_rank-1 the reduction axes.
 * Only nodes below a FOLD may have non-zero strides on reduction axes.
 */
typedef struct mdim_node {
    int32_t kind;      /* mdim_node_kind */
    int32_t dtype;     /* result dtype of this node */
    int32_t op;        /* BINARY: mdim_binary_op; UNARY: mdim_unary_op; FOLD: mdim_binary_op */
    int32_t n_comp;    /* GATHER: number of index components (= children); DIAG: number of pairs; FOLD: 2 = (init, body) children */
    int32_t src_dtype; /* UNARY/CAST: dtype of the operand */
    int32_t n_peers;   /* LEAF/GATHER: 0/1 = `data` is one buffer; k>1 = the source Array is split into k
                          equal blocks of `peer_block` elements along its linear index, block p at
                          peer[p] (peer-mapped HBM of the other GPUs of the box, read over NVLink).
                          A sharded LEAF is what a transpose of a row-sharded Array reads: the all-to-all
                          happens inside the transpose kernel, tile by tile */
    const void* data;  /* LEAF/GATHER: device base pointer of the source Array's items */
    int64_t offset;    /* LEAF/GATHER/IOTA: constant element offset (Row/Column/fixed coords) */
    int64_t stride[MDIM_MAX_RANK];  /* LEAF/GATHER/IOTA: elements per step of each iteration axis;
                                       0 = operand lacks the axis (Broadcast, src/broadcast.rs:46-60) */
    int64_t gstride[MDIM_MAX_RANK]; /* GATHER: elements per unit of index component c */
    uint64_t bound[MDIM_MAX_RANK];  /* GATHER: size of component c; idx >= bound is MDIM_ERR_OOB */
    int32_t axis_a[MDIM_MAX_RANK];  /* DIAG pair p: iteration axis on the left ... (CONCAT: [0] = the axis) */
    int32_t axis_b[MDIM_MAX_RANK];  /* ... equals iteration axis on the right PLUS (int64_t)axis_c[p] (a shard of a
                                       Diagonal: its block starts at a non-zero coordinate), or, if axis_b[p] < 0, */
    uint64_t axis_c[MDIM_MAX_RANK]; /* ... equals the constant axis_c[p] (a Row/Column of a Diagonal);
                                       CONCAT: [0] = length of V along the axis; W's strides are already
                                       expressed against the concatenated coordinate (offset shifted) */
    mdim_scalar imm;                /* CONST value; DIAG `zero`; FOLD init */
    const void* peer[MDIM_MAX_PEERS];
    uint64_t peer_block;
} mdim_node;

typedef struct mdim_expr {
    int32_t abi_version; /* MDIM_ABI_VERSION */
    int32_t rank;        /* output leaf axes (0 = a single element) */
    int32_t red_rank;    /* reduction leaf axes, iterated sequentially last-fastest under a FOLD */
    int32_t n_nodes;
    uint64_t length[MDIM_MAX_RANK]; /* rank + red_rank entries */
    const mdim_node* nodes;         /* caller-owned, borrowed for the duration of the call */
} mdim_expr;

/* Details of the first (lowest output position) failing element of the last failed collect. */
typedef struct mdim_error_info {
    int32_t status;    /* mdim_status */
    int32_t node;      /* index of the node that failed, -1 if not attributable */
    uint64_t position; /* linear output position (to_usize order) of the failing element */
    uint64_t value;    /* OOB: the offending index component; ARITH: the divisor bits */
    uint64_t bound;    /* OOB: the size it was checked against */
    int32_t component; /* OOB: which index component */
    int32_t reserved;
    char message[160]; /* reference-style panic text, e.g. "Index 7 is out of bounds for size 3" */
} mdim_error_info;

typedef struct mdim_ctx mdim_ctx;

/* flags of mdim_collect */
#define MDIM_COLLECT_ASYNC 1u      /* do not synchronise; errors surface at mdim_sync */
#define MDIM_COLLECT_NO_FASTPATH 2u /* force the general rank-N evaluator (testing/benchmarks) */
#define MDIM_COLLECT_NO_STATIC 4u   /* force the interpreted op-tree (testing/benchmarks) */
#define MDIM_COLLECT_NO_JIT 8u      /* do not specialise unlisted op trees at run time (NVRTC) */

#ifndef __CUDACC_RTC__ /* (the declarations below are host functions; NVRTC compiles this header too) */
/* ---- context ---------------------------------------------------------------------------------- */
int mdim_init(int device, mdim_ctx** ctx);
int mdim_shutdown(mdim_ctx* ctx);
/* Launch on a caller-owned cudaStream_t (e.g. torch's current stream); NULL = the context's own.  It first waits for every collect
 * on the old stream, so a context's collects never run on two streams at once (the scratch of the few-output integer folds,
 * k_fold_split, relies on this: one context, one stream at a time). */
int mdim_set_stream(mdim_ctx* ctx, void* cuda_stream);
/* The stream collects are launched on (a cudaStream_t): the context's own unless mdim_set_stream replaced it.  Record
 * CUDA events on it to time collects.  On its OWN stream the context knows every kernel in flight, so a collect whose
 * operands and output are untouched by the kernels still running starts before they finish (dependency-aware
 * programmatic launch, csrc/launch.cuh); on a caller-owned stream every kernel waits for its predecessor. */
int mdim_get_stream(mdim_ctx* ctx, void** cuda_stream);
int mdim_sync(mdim_ctx* ctx); /* waits for the stream; returns the deferred status of async collects */
int mdim_last_error(mdim_ctx* ctx, mdim_error_info* info);
const char* mdim_status_string(int status);
uint64_t mdim_launch_count(mdim_ctx* ctx); /* kernels launched by this library so far */
/* The kernel the LAST collect launched: a pre-built one ("k_eval<SigMulAddCF32>...", "k_transpose_tma", "k_fold_regs"), or
 * "mdim_jit_kernel[ops]" / "mdim_jit_kernel[ops+shape]" when the chain was specialised at run time.
 * NVRTC (libnvrtc, part of the CUDA toolkit) is OPTIONAL: without it, or with MDIM_COLLECT_NO_JIT, chains outside the
 * pre-built signature table run through the depth-specialised interpreter of the same evaluator (about 0.3x of the
 * specialised rate), and rank >= 2 chains keep run-time strides (config 5: 0.61 instead of 0.93 of 8 TB/s). */
int mdim_last_kernel(mdim_ctx* ctx, char* buf, size_t buf_len);
int mdim_device_info(mdim_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, size_t* hbm_bytes);

/* ---- device-resident boxed buffer: the `Box<[T]>` of Array (src/array.rs:5-8) ------------------ */
int mdim_buf_alloc(mdim_ctx* ctx, size_t bytes, void** dptr);
int mdim_buf_free(mdim_ctx* ctx, void* dptr);
int mdim_upload(mdim_ctx* ctx, void* dst_device, const void* src_host, size_t bytes);
int mdim_download(mdim_ctx* ctx, void* dst_host, const void* src_device, size_t bytes);
int mdim_host_alloc(mdim_ctx* ctx, size_t bytes, void** hptr); /* pinned host memory */
int mdim_host_free(mdim_ctx* ctx, void* hptr);

/* ---- the hot path ------------------------------------------------------------------------------ */
/* View::collect (src/view.rs:146-150): materialise `e` into the dense row-major buffer `out`
 * (device memory, prod(length[0..rank)) elements of the root dtype, never aliasing an input).
 * `out` must be aligned to its element size (else MDIM_ERR_INVALID); 16-byte alignment enables 128-bit stores and
 * the TMA transpose, 32-byte alignment the 256-bit stores (cudaMalloc gives 256).  An output that is only
 * element-aligned (a slice of a caller's tensor) is written with scalar stores. */
int mdim_collect(mdim_ctx* ctx, const mdim_expr* e, void* out_device, uint32_t flags);

/* View::collect of a tuple-typed view: `e`'s root is an MDIM_NODE_TUPLE with n_outs children; outs_device[c] receives the run
 * of scalar leaf c (see "layout of tuple-typed Arrays").  One kernel launch; same flags, errors and alignment rules. */
int mdim_collect_tuple(mdim_ctx* ctx, const mdim_expr* e, void* const* outs_device, int n_outs, uint32_t flags);

/* Same, but every LEAF/GATHER `data` pointer and `out` are HOST buffers: uploads, collects and
 * downloads, chunked along the outermost axis and pipelined over copy/compute streams when the
 * expression shards there.  This is the call a host-array user (`Array::new(..)` → collect →
 * `to_raw()`, src/array.rs:28-30,54) makes, and what bench.py's e2e figure times. */
int mdim_collect_host(mdim_ctx* ctx, const mdim_expr* e, void* out_host, uint32_t flags);

/* Which kernel the planner picks for `e` (e.g. "stream.static[mul_add_c] v4"); for tests, bench. */
int mdim_plan_describe(mdim_ctx* ctx, const mdim_expr* e, uint32_t flags, char* buf, size_t buf_len);
/* The same planning step without a device (ctx may be NULL): usable on a CPU-only box. */
int mdim_plan_describe_nodevice(const mdim_expr* e, uint32_t flags, char* buf, size_t buf_len);

/* ---- peer memory for sharded gather sources (one process per GPU, NVLink/NVSwitch) ------------- */
#define MDIM_IPC_HANDLE_BYTES 64
int mdim_ipc_export(mdim_ctx* ctx, void* dptr, uint8_t handle[MDIM_IPC_HANDLE_BYTES]);
int mdim_ipc_open(mdim_ctx* ctx, const uint8_t handle[MDIM_IPC_HANDLE_BYTES], void** dptr);
int mdim_ipc_close(mdim_ctx* ctx, void* dptr);

/* ---- multi-GPU: one process per GPU, one context per process (SURVEY.md §8e) -----------------------------------------
 * The reference has no distributed layer; this is the surface a sharded `DeviceArray` needs so that the Rust host (or
 * the C++ / Python mirrors) can partition Arrays along the outermost index WITHOUT any other runtime:
 *   - a communicator (NCCL, loaded at run time; rank 0 makes the id, the caller ships its 128 bytes to the other
 *     ranks by any means it has — a file, a socket, MPI, an environment variable);
 *   - the two collectives the north star names, on the context's stream: all-gather of a sharded compose() source
 *     (src/view.rs:897-912) and all-reduce of the partial folds over a sharded axis (src/view.rs:617-622);
 *   - the peer table: every rank's block mapped into every process (CUDA IPC), for mdim_node.peer[] — the gather,
 *     transpose and fold kernels then read the owning GPU's HBM over NVLink inside the kernel, no collective.
 * All of these are COLLECTIVE calls: every rank of the communicator makes them in the same order. */
#define MDIM_COMM_ID_BYTES 128
int mdim_comm_unique_id(uint8_t id[MDIM_COMM_ID_BYTES]);                                 /* rank 0 */
int mdim_comm_init(mdim_ctx* ctx, int rank, int world, const uint8_t id[MDIM_COMM_ID_BYTES]);
int mdim_comm_destroy(mdim_ctx* ctx);
int mdim_comm_info(mdim_ctx* ctx, int* rank, int* world, int* nccl_version);
int mdim_allgather(mdim_ctx* ctx, const void* send_device, void* recv_device, size_t block_bytes); /* async, rank-major */
int mdim_allreduce(mdim_ctx* ctx, void* data_device, size_t n, int dtype, int op);       /* async, in place; op: MDIM_ADD,
                                                                                             MDIM_MUL, MDIM_REDUCE_MIN/MAX */
int mdim_barrier(mdim_ctx* ctx);                                                          /* + waits for the stream */
int mdim_peer_table(mdim_ctx* ctx, void* local_device, size_t block_bytes, void* peers[MDIM_MAX_PEERS]);
int mdim_peer_table_close(mdim_ctx* ctx);                                                 /* unmaps every peer block */
/* Fold over the SHARDED (outermost) axis, BIT-IDENTICAL to the reference's sequential chain (src/view.rs:617-622, 250-252):
 * `local_rows` = this rank's rows (dense row-major n_rows_local x n_cols, device memory), ranks in index order;
 * out[c] = (((init (op) x[0][c]) (op) x[1][c]) ... ) over ALL ranks' rows, on EVERY rank.  One fused kernel per GPU: the running
 * values travel rank to rank through peer-mapped HBM, pipelined over column slices (csrc/k_fold_ring.cu) — no all-reduce, no
 * reassociation.  op: MDIM_ADD, SUB, MUL, AND, OR, XOR; 4- and 8-byte dtypes; n_cols <= 2^20 per call, rows 16-byte aligned.
 * Asynchronous on the context's stream; mdim_fold_sharded_axis_status reports (and clears) a peer that never arrived: the kernels' waits
 * are bounded (~2 s), the result is then garbage, and the ranks' launch counters no longer agree — destroy and re-create the communicator
 * on every rank before folding over a sharded axis again (tests/test_comm_multi_gpu.py::test_a_missing_peer_is_an_error_not_a_hung_gpu). */
int mdim_fold_sharded_axis(mdim_ctx* ctx, const void* local_rows, uint64_t n_rows_local, uint64_t n_cols, int dtype, int op, mdim_scalar init,
                           void* out_device);
int mdim_fold_sharded_axis_status(mdim_ctx* ctx);
/* The all-reduce route of the same fold (SURVEY.md 8e) as ONE fused kernel per GPU (csrc/k_fold_xchg.cu), no NCCL call:
 * P_r = rank r's rows folded sequentially (rank 0 starts from `init`, the others from the operator's identity: 0, 1, all-ones, and
 * -0.0 for a float sum); out[c] = ((P_0 (op) P_1) (op) P_2) ... (op) P_{N-1} on EVERY rank, combined in rank order inside the kernel
 * from flag-in-data packets written into peer-mapped HBM.  Bit-identical to the reference for integer and bitwise folds; a float
 * fold is reassociated at the rank boundaries only: deterministic, as accurate as the reference's own order, and ~1e-6 relative away
 * from it over 1024 f32 terms (2 % of the outputs of a (1024, 2^18) sum by more than 1e-6, at most 2.2e-6: the same as ncclAllReduce).  op: MDIM_ADD, MUL, AND, OR, XOR; 4- and
 * 8-byte dtypes; rows and out 16-byte aligned, row length a multiple of 16 bytes.  Asynchronous; errors as above. */
int mdim_fold_sharded_axis_blocked(mdim_ctx* ctx, const void* local_rows, uint64_t n_rows_local, uint64_t n_cols, int dtype, int op,
                                   mdim_scalar init, void* out_device);

/* Run-time specialisation (NVRTC) of `e`'s op tree, compile step only: needs no GPU.  0 = compiles for
 * sm_100a; MDIM_ERR_UNSUPPORTED = NVRTC not installed or the plan has a pre-built kernel; `log` gets details. */
int mdim_jit_check_nodevice(const mdim_expr* e, uint32_t flags, char* log, size_t log_len);

int mdim_abi_version(void);
#endif /* __CUDACC_RTC__ */

#ifdef __cplusplus
}
#endif
#endif /* MDIM_H */
