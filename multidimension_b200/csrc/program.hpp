// program.hpp — the flattened device program a View chain is lowered to.
//
// The host planner (plan.cpp) turns the C-ABI descriptor (include/mdim.h: mdim_expr, a post-order
// node array in position space) into this POD, which is passed BY VALUE as a __grid_constant__
// kernel parameter (constant bank; ~3.3 KB).  The kernels (kernels.cuh) execute it either through
// the depth-specialised interpreter or through a compile-time signature (static op tree).
//
// Reference semantics each instruction carries are cited in exec.cuh next to its implementation.
#pragma once
#include <stdint.h>

#include "../../include/mdim.h"

namespace mdim {

constexpr int kMaxRank = MDIM_MAX_RANK;
constexpr int kMaxInstr = 56;
constexpr int kMaxAddr = 12;
constexpr int kMaxPred = 16;
constexpr int kMaxComp = 4;
constexpr int kMaxDepth = 8;  // deepest value stack any instantiation supports

enum Opc : uint8_t {
    OPC_LEAF_VEC = 0,   // contiguous along the vector axis, aligned: 128-bit loads
    OPC_LEAF_BCAST,     // stride 0 along the vector axis: one scalar load, replicated
    OPC_LEAF_STRIDED,   // anything else: V scalar loads
    OPC_IOTA,           // linear combination of coordinates
    OPC_CONST,
    OPC_UNARY,
    OPC_BINARY,
    OPC_MASK,           // set the lane-active mask from pred[slot .. slot+n)  (n = 0: all active)
    OPC_SELECT,         // Diagonal: keep TOS where pred[slot .. slot+n) holds, else imm
    OPC_SELECT2,        // Concat: pops W (TOS) and V; keeps V where pred[slot] holds, else W
    OPC_GATHER,         // pops aux index components, bounds-checks, loads
    OPC_FOLD_BEGIN,     // push acc = imm, reset reduction coordinates
    OPC_FOLD_STEP,      // acc = acc (op) TOS; advance reduction coords; loop to pc = slot
    OPC_COUNT
};

struct Instr {  // 16 bytes
    uint8_t opc;
    uint8_t dtype;  // result dtype (mdim_dtype)
    uint8_t op;     // mdim_binary_op / mdim_unary_op
    uint8_t aux;    // UNARY: source dtype; BINARY/FOLD_STEP: rhs dtype; GATHER: n_comp;
                    // LEAF_VEC: 1 = the operand is re-read (broadcast along some axis): allocate in L1
    uint16_t slot;  // LEAF/IOTA/GATHER: addr index; MASK/SELECT: first pred; FOLD_STEP: loop pc
    uint16_t n;     // MASK/SELECT: pred count; BINARY/GATHER/FOLD_STEP: source node (error reports)
    uint64_t imm;   // CONST value bits; SELECT zero; FOLD_BEGIN init
};

struct Addr {
    const void* ptr;
    int64_t offset;             // elements
    int64_t stride[kMaxRank];   // elements per unit of each (coalesced) iteration axis
    int64_t inner;              // stride along the innermost OUTPUT axis (the vector axis)
    int64_t rstride;            // stride along the FASTEST reduction axis (walked by ThreadState::rk, not by c[])
    int64_t gstride[kMaxComp];  // GATHER: elements per unit of index component
    uint64_t bound[kMaxComp];   // GATHER: size of index component
    int32_t n_peers;            // GATHER over peer-mapped shards (see mdim_node.n_peers)
    int32_t pad;
};

struct Pred {  // sum_a coef[a] * coord[a] (+ lane * lane_coef)  ==  rhs   (cmp 0: Diagonal)
               //                                              <   rhs   (cmp 1: Concat, V side)
               //                                              >=  rhs   (cmp 2: Concat, W side)
    int32_t coef[kMaxRank];
    int32_t lane_coef, cmp;  // lane_coef: coef of the innermost output axis
    int32_t rcoef, pad;      // coef of the FASTEST reduction axis: its coordinate is ThreadState::rk, not c[] (like Addr::rstride)
    int64_t rhs;
};

struct PeerTab {
    const void* peer[MDIM_MAX_PEERS];
    uint64_t block;
};

enum ProgFlags : uint32_t {
    PF_EXPLAIN = 1u,  // single-lane rerun that records mdim_error_info details
    PF_VEC256 = 2u,   // every vector operand and the output are 32-byte aligned: 256-bit loads / stores
    PF_GATHER_BIG = 8u,  // a gathered source spans more than kGatherBigBytes: 64-byte L2 fetches (exec.cuh: ld32_big)
    PF_NOWAIT = 4u,   // no buffer of this launch is touched by a kernel still in flight: skip griddepcontrol.wait (launch.cuh)
};

struct Program {
    // Axis numbering of every per-axis array below: the output axes INNERMOST FIRST (axis 0 is the
    // vector axis, axis rank-1 the outermost), then the reduction axes in iteration order.
    int32_t rank;      // coalesced output axes
    int32_t red_rank;  // coalesced reduction axes
    int32_t n_instr, n_addr, n_pred;
    int32_t out_dtype;
    int32_t n_out;            // 1, or the number of scalar leaves of a tuple-typed root (MDIM_NODE_TUPLE): value k of the final stack goes to out k
    int32_t out_dtypes[MDIM_MAX_OUTS];
    void* out_more[MDIM_MAX_OUTS - 1];  // run-time: the output runs 1.. (run 0 is the kernel's `out` argument)
    int32_t vec;  // lanes per vector along the innermost output axis (program axis 0)
    int32_t pad0; // keeps length[] and the fields after it at their offsets (moved, the evaluators compile one constant load differently)
    uint32_t flags;
    uint64_t length[kMaxRank];  // coalesced lengths: out axes then reduction axes (elements)
    uint64_t dec_len[kMaxRank];   // decode length of axis a: innermost out axis in vectors; 1 if not an out axis
    uint32_t dec_scale[kMaxRank]; // vec for the innermost out axis, else 1
    uint32_t div_mul[kMaxRank];   // magic multiplier/shift for division by dec_len[a] (32-bit path)
    uint32_t div_shr[kMaxRank];
    uint64_t n_vec;             // total output vectors = prod(out lengths) / vec
    uint64_t red_count;         // prod(reduction lengths)
    uint64_t red_fast_len;      // length of the fastest reduction axis (its entry in length[] is 1, its stride[] entries 0)
    uint64_t explain_pos;       // PF_EXPLAIN: output position whose failure details to record
    Instr instr[kMaxInstr];
    Addr addr[kMaxAddr];
    Pred pred[kMaxPred];
    PeerTab peers;
};

// Device-side error word: kernels atomicMin the linear output position of a failing element;
// the host then reruns that one element with PF_EXPLAIN to fill the details.
struct ErrWord {
    unsigned long long pos;  // ~0ull = no error
    int32_t status, node, component, pad;
    unsigned long long value, bound;
};

// ---- planning result ------------------------------------------------------------------------
enum KernelKind : int32_t {
    KK_EMPTY = 0,      // zero-length output: nothing to launch
    KK_GENERIC = 1,    // rank-N evaluator (k_eval)
    KK_STREAM = 2,     // rank-<=1 contiguous: k_eval with the decode compiled out
    KK_TRANSPOSE = 3,  // tiled smem transpose of one leaf (k_transpose)
    KK_FOLD_ROWS = 4,  // last-axis sequential fold (+ fused broadcast epilogue) (k_fold_rows)
    KK_FOLD_COLS = 5,  // sequential fold over an OUTER axis of one leaf whose result is contiguous: a column walk (k_fold_cols)
    KK_FOLD_SPLIT = 6, // integer fold with few outputs and a long reduction: the reduction cut into chunks over the whole GPU (k_fold_split)
};

// The register-staged transpose's tile (k_transpose.cu): 16-byte chunks along A x source rows, 256-byte runs both ways.
// Measured on B200: 32 x 128 equal at 16384^2 (6.31 vs 6.32 TB/s) and slower at 4096^2 (5.25 vs 5.67), as were 32 x 64
// and 16 x 128 (5.1 TB/s).
constexpr int kTrTileChunks = 16, kTrTileRows = 64;

struct TransposePlan {
    const void* src;
    int32_t esize;
    int64_t src_offset;
    // out index space: batch axes (coalesced) x [A] x mid axes x [B] where B is the out-inner axis
    // (out stride 1) and A is the axis whose SOURCE stride is 1.
    int32_t n_batch;             // number of remaining axes (all but A and B)
    uint64_t batch_len[kMaxRank];
    int64_t batch_src_stride[kMaxRank];
    int64_t batch_out_stride[kMaxRank];
    uint64_t len_a, len_b;       // extents of A and B
    int64_t src_stride_b;        // source stride along B (A has source stride 1)
    int64_t out_stride_a;        // out stride along A (B has out stride 1)
    uint64_t tiles_a, tiles_b, n_tiles;
    // Source sharded over peer GPUs (mdim_node.n_peers on the LEAF): element e of the whole Array lives at
    // peer[e / peer_block] + (e % peer_block).  The kernel reads the owning peer's HBM over NVLink, so the
    // all-to-all a row-sharded transpose implies happens inside the tile loads.
    int32_t n_peers;
    float peer_inv;              // 1 / peer_block (quotient estimate, corrected exactly in the kernel)
    uint64_t peer_block;
    const void* peer[MDIM_MAX_PEERS];
    int32_t nowait;              // set per launch by its launcher: see launch.cuh
};

struct FoldRowsPlan {
    const void* src;
    int64_t src_offset;
    uint64_t n_rows;   // number of independent rows
    uint32_t row_len;  // reduction length (contiguous)
    int32_t op;        // mdim_binary_op
    int32_t dtype;
    uint64_t init;
    // epilogue: 0 = emit the fold (one value per row); 1 = out[r][k] = src[r][k] (eop) g(fold[r])
    int32_t epilogue;
    int32_t eop;          // binary op of the epilogue, src on the left
    int32_t post_op;      // optional binary op applied to the fold before the epilogue (e.g. DIV)
    int32_t has_post;
    uint64_t post_imm;    // ... with this constant on the right
    int32_t nowait;       // set per launch by its launcher: see launch.cuh
};

struct FoldColsPlan {
    const void* src;      // first byte of row 0 (offset applied)
    uint64_t n_rows;      // reduction length: rows walked in index order
    uint64_t row_bytes;   // bytes of one row that take part (= bytes of the result; multiple of 16)
    uint64_t pitch_bytes; // bytes between consecutive rows (multiple of 16)
    uint64_t n_batch;     // independent blocks (an axis OUTSIDE the folded one); their results lie back to back
    uint64_t batch_pitch_bytes;  // bytes between consecutive blocks (multiple of 16)
    int32_t op, dtype;
    uint64_t init;
};

// k_fold_split.cu: an integer fold whose operator is associative and commutative (wrapping Add, Mul, BitAnd, BitOr, BitXor; Sub as
// init - sum), so any order of combination gives the reference's bits.  Taken for at most kSplitMaxOuts outputs and a reduction
// of at least kSplitMinRed elements (kSplitMaxCols outputs when they are columns): there the other routes leave most of the GPU
// idle, one thread or a few walking each output.  Measured on one B200 (1000 W), u32 sums (profiles/r3_fold_split_bench.txt):
// the split fold wins at every reduction length measured (down to 2^12) for up to 16384 runs and up to 1024 columns, and loses
// at 4096 columns (71 against 264 GB/s for k_fold_cols: the finishing CTA's combine caps the chunks of a wide row).
constexpr uint64_t kSplitMaxOuts = 4096, kSplitMaxCols = 1024, kSplitMinRed = 1ull << 12;
enum SplitLayout : int32_t { SPLIT_RUNS = 0, SPLIT_COLS = 1 };
struct FoldSplitPlan {
    const void* src;        // element 0 of the walk (the leaf's offset and any flipped reduction axis applied)
    int32_t layout;         // SPLIT_RUNS: each output reduces one run of `red` contiguous elements
                            // SPLIT_COLS: each output is a column; `cols` contiguous columns per row, rows `pitch` apart
    int32_t op;             // MDIM_ADD, SUB, MUL, AND, OR, XOR
    int32_t dtype, src_dtype;  // the fold's dtype; the leaf's (a CAST body converts between them)
    int32_t slot_bytes;     // 4 or 8: the accumulator width (the fold's dtype, U8 widened to 4)
    int32_t nowait;         // set per launch by its launcher: see launch.cuh
    uint64_t init;          // bits of the immediate init
    uint64_t red;           // RUNS: elements per run; COLS: rows
    uint64_t n_out;         // outputs, written contiguously
    uint64_t out_len[2];    // RUNS: output o = i0 * out_len[1] + i1 starts at i0 * out_stride[0] + i1 * out_stride[1] (elements)
    int64_t out_stride[2];
    uint64_t cols, n_batch; // COLS: output o = b * cols + c reads b * batch_stride + r * pitch + c (elements)
    int64_t pitch, batch_stride;
};

// Memory a launch reads (api.cu adds the output and decides whether the kernel may skip griddepcontrol.wait).
constexpr uint64_t kGatherBigBytes = 1ull << 30;  // ~8x the 126 MB L2: below that the plain load's L2 hits win (probe)
constexpr int kMaxRanges = 24;
struct MemRange { uint64_t lo, hi; };  // [lo, hi) bytes

// Internal planning flag (never part of the C ABI's MDIM_COLLECT_* set): the output buffer is only element-aligned
// (e.g. a slice of someone else's tensor), so every store must be scalar and the vector-store fast paths are off.
constexpr uint32_t kPlanScalarOut = 0x10000u;

// k_fold_ring.cu: the bit-exact fold over the sharded axis (one fused compute + exchange kernel per GPU)
struct FoldRingArgs {
    uint64_t n_rows, n_cols;   // this rank's rows x the (unsharded) columns
    int32_t dtype, op, esize, rank, world;
    uint32_t epoch;            // launch counter of the communicator: every 16-byte line carries it, so the areas never need resetting
    uint64_t init;             // bits of the fold's initial value (rank 0 starts from it)
    const void* inbox;         // this GPU's inbox: running values written by rank - 1 as {word, epoch, word, epoch} lines (2 x the data bytes)
    void* next_inbox;          // rank + 1's inbox (peer-mapped)
    void* result[MDIM_MAX_PEERS];        // every rank's result area (the last rank writes the finished slices into all of them, same lines)
    void* out;
    uint32_t* error;           // set to 1 when a peer did not arrive in time
};

// k_fold_xchg.cu: fold over the sharded axis as per-rank partial folds + an in-kernel all-reduce in RANK ORDER (one fused
// compute + exchange kernel per GPU; flag-in-data packets through peer-mapped HBM, no fence, no NCCL call)
struct FoldXchgArgs {
    uint64_t n_rows, row_bytes, pitch_bytes;  // this rank's rows; bytes of one row that take part (multiple of 16); bytes between rows
    uint64_t n_batch, batch_pitch_bytes;      // one-GPU form only: independent (rows x columns) blocks and the bytes between them
    int32_t rank, world;
    uint32_t epoch;            // launch counter: the packets carry it, so the areas never need resetting
    int32_t wide;              // rows and pitch are 32-byte aligned: 256-bit loads
    int32_t one_shot;          // every rank sends to every rank and combines (one hop) instead of owners (two hops)
    int32_t nowait;            // one-GPU form only: the launch is independent of its predecessors (launch.cuh)
    uint32_t slot;             // epoch & 1: two sets of areas alternate, so a rank one launch ahead cannot overwrite unread packets
    uint64_t start;            // bits of the value this rank's chain starts from (rank 0: init; others: the operator's identity)
    uint64_t cap_words;        // 32-bit words of one (slot, source rank) area
    const void* rows;
    char* area[MDIM_MAX_PEERS];  // every rank's packet area (peer-mapped; area[rank] is local)
    void* out;
    uint32_t* error;           // set to 1 when a peer's packets did not arrive in time
};

struct Plan {
    int32_t kind;
    uint32_t flags;      // the MDIM_COLLECT_* flags the plan was made with
    int32_t slot_bytes;  // 4 or 8: width of the value-stack slots
    int32_t vec;
    int32_t wide;        // 64-bit coordinates/strides
    int32_t n_axes;      // rank + red_rank after canonicalisation (selects the MAXR instantiation)
    int32_t vec256_ok;   // every LEAF_VEC operand is 32-byte aligned (the output is checked at launch)
    int32_t max_depth;
    int32_t variant;     // the k_eval instantiation that serves the evaluator's program (index into kEvalVariants), -1 = none
    int32_t static_id;   // = variant when that instantiation runs a pre-built signature, else -1 (interpreted)
    uint64_t out_elems;
    int32_t out_esize;
    int32_t n_out;                        // > 1: tuple-typed root
    int32_t out_esizes[MDIM_MAX_OUTS];
    Program prog;
    TransposePlan tr;
    FoldRowsPlan fr;
    FoldColsPlan fc;
    FoldSplitPlan fs;
    char sig[kMaxInstr * 4 + 4];  // signature bytes (opc,dtype,op,aux per instruction)
    int32_t sig_len;
    char describe[192];
    MemRange in_range[kMaxRanges];  // every LEAF / GATHER source (and each peer block) as a byte range
    int32_t n_in_ranges;            // -1: not tracked (too many operands): the launch waits for its predecessor
};

#ifndef __CUDACC_RTC__  // host-side declarations (this header is also compiled by NVRTC, see jit.cu)
int plan_expr(const mdim_expr* e, uint32_t flags, Plan* plan, char* why, size_t why_len);
// plan_expr for a collect into the output runs outs[0 .. n_outs) (one per scalar leaf of a TUPLE root, else one): checks each run
// (not null, aligned to its element), plans again with scalar stores when a run is only element-aligned, and fills out_more[]
int plan_collect(const mdim_expr* e, uint32_t flags, void* const* outs, int n_outs, Plan* plan, char* why, size_t why_len);
int dtype_size(int dt);
const char* status_string(int st);
// mdim_error_info for a device-side failure at output position `pos`, from the error word of its PF_EXPLAIN rerun
void explain_failure(const ErrWord& w, uint64_t pos, mdim_error_info* info);

// Every k_eval instantiation (kernels.cuh), as the planner selects among them: the variants_*.inc lists in the order s32 static,
// s64 static, s32 interp, s64 interp, which is also the order of the kernels k_eval_*.cu export.
struct SigInstr;
struct EvalVariant {
    const char* name;
    int slot_bytes, vec, max_depth, wide, maxr;  // maxr: iteration axes walked (1 = contiguous stream)
    const SigInstr* sig;  // nullptr = interpreter
    int sig_n;
};
extern const EvalVariant kEvalVariants[];
extern const int kNumEvalVariants;
// the instantiation's template arguments, e.g. k_eval<SigSubBcastF32,s32,v8,d4,r3> or k_eval<interp,s64,v1,d8,wide,r8>
void eval_variant_name(int variant, char* buf, size_t len);

// Per iteration axis, the coordinates [lo, hi) over which a node is evaluated, and the elements [lo, hi) an operand reaches over
// them, relative to its data pointer (offset + sum of stride * coordinate, plus the gathered components over [0, bound)).
struct AxisRange { uint64_t lo[MDIM_MAX_RANK], hi[MDIM_MAX_RANK]; };
struct ElemRange { int64_t lo, hi; };
// the whole axes at the root, narrowed under a CONCAT: its V side sees [0, len(V)), its W side [len(V), end)
void node_axis_ranges(const mdim_expr* e, AxisRange* out);  // out: e->n_nodes entries
ElemRange operand_reach(const mdim_expr* e, const mdim_node& n, const AxisRange& r, int first_axis);  // axes [first_axis, rank + red_rank)

// jit.cu: a kernel specialised at run time for the plan's op sequence, or nullptr (use the interpreter)
// explain: the single-element rerun of a failed collect; it reuses a shape kernel already built but neither counts towards nor triggers one
void* jit_kernel_for(const Plan& p, int* level = nullptr, bool explain = false);  // level: 0 none, 1 specialised on the op sequence, 2 on ops AND shape

// NVRTC half of jit_kernel_for alone (needs no GPU): 0 = the specialisation compiles for sm_100a
int jit_compile_check(const Plan& p, char* log, size_t log_len);
#endif

}  // namespace mdim
