/*
 * genfer_taylor.h -- C ABI of libgenfer_taylor.so, the B200 (sm_100a) implementation of genfer's
 * dense truncated Taylor arithmetic for the f64 Number path.
 *
 * The reference (fzaiser/genfer, pure Rust) has no FFI layer: its boundary for this path is the
 * generic value type `TaylorPoly<T: Number>` (src/multivariate_taylor.rs:13-19) with
 * `impl Add/Sub/Mul/Div/Neg` (:854-1237) plus ~25 inherent methods, and the univariate
 * `TaylorExpansion<T>` (src/univariate_taylor.rs:9-13, `impl Number` :150-211).  Each entry point
 * below replaces one of those for T = F64 and cites it.  A Rust `extern "C"` shim that binds these
 * (rust/genfer-taylor-sys) and the patch to multivariate_taylor.rs are shown in INTEGRATION.md.
 *
 * Conventions
 *  - Plain pointers and sizes only.  Handles are opaque.  All functions return a gtp_status
 *    (0 = ok); `gtp_last_error(ctx)` gives the message.  Where the reference would panic
 *    (assert!/index out of bounds) the call returns GTP_ERR_INDEX and the Rust shim panics.
 *  - Element type is IEEE-754 binary64.  Buffers are dense, row-major over the STORED shape
 *    (`coeffs.shape()`), last variable fastest, base pointer >= 256-byte aligned.  The conceptual
 *    truncation `degrees_p1` is host metadata; GTP_UNBOUNDED (= usize::MAX) means "exact
 *    polynomial, no truncation" (generating_function.rs:485, :569).
 *  - Value semantics like the reference: every operation returns a NEW handle and never mutates
 *    or aliases-for-write its inputs (buffers are immutable and reference counted, so clone is O(1);
 *    the reference deep-copies, multivariate_taylor.rs:10-12).  The caller frees every handle.
 *  - One context = one CUDA device + one stream.  Calls on one context are not re-entrant
 *    (the reference is single threaded, src/main.rs:96-106).  Launches are asynchronous; only the
 *    scalar readers and gtp_to_host synchronise.  Operator dispatch needs a few data-dependent
 *    predicates (is_zero / is_one / extract_linear, multivariate_taylor.rs:1021-1061): these are
 *    evaluated by a device kernel and cached per handle.
 *  - There is NO CPU fallback: if no CUDA device is present gtp_ctx_create fails with GTP_ERR_CUDA.
 */
#ifndef GENFER_TAYLOR_H
#define GENFER_TAYLOR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GTP_UNBOUNDED UINT64_MAX /* Rust usize::MAX */
#define GTP_MAX_NDIM 24

typedef enum gtp_status {
  GTP_OK = 0,
  GTP_ERR_INDEX = 1, /* the reference's assert!/panic on a bad variable / order / index   */
  GTP_ERR_SHAPE = 2, /* violated shape/degree invariant (check_invariants, :23-31)         */
  GTP_ERR_OOM = 3,   /* device allocation failed                                           */
  GTP_ERR_CUDA = 4,  /* CUDA runtime / launch error, or no device                          */
  GTP_ERR_ARG = 5    /* null pointer, ndim > GTP_MAX_NDIM, ...                              */
} gtp_status;

typedef struct gtp_ctx gtp_ctx;   /* device + stream + stream-ordered pool + pinned read-back page */
typedef struct gtp_poly gtp_poly; /* TaylorPoly<F64>  (multivariate_taylor.rs:13-19)              */
typedef struct gtu_series gtu_series; /* TaylorExpansion<F64> (univariate_taylor.rs:9-13)         */

/* ---- context ------------------------------------------------------------------------------- */
/* `cuda_stream` may be NULL (the context creates its own non-blocking stream) or an existing
 * cudaStream_t (e.g. torch's current stream) to interleave with the caller's work. */
int gtp_ctx_create(int device, void* cuda_stream, gtp_ctx** out);
void gtp_ctx_destroy(gtp_ctx* ctx);
const char* gtp_last_error(gtp_ctx* ctx);
int gtp_ctx_synchronize(gtp_ctx* ctx);
/* Returns the context's cached free device blocks to the driver (the context keeps freed blocks in a PRIVATE
 * stream-ordered pool -- the device's default pool is never modified -- so that other allocators of the process
 * are only affected by memory this context actually holds).  Synchronises. */
int gtp_ctx_trim(gtp_ctx* ctx);
void* gtp_ctx_stream(gtp_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t gtp_ctx_launch_count(gtp_ctx* ctx);
/* tuning knob: 0 = always use the reference-order product kernel (bit-identical products, Horner loops and 2-axis log / exp;
 * general N-D division and N-D log stay tolerance-level: their wavefront / descending-row summation order is not the reference's),
 * 1 = pick the fastest applicable kernel (default: DFMA kernels from 2^20 MACs), 2 = use the DFMA kernels even for
 * tiny products (tests).  A/B bits: +4 and +8 are ignored (retired variants of the blocked kernel's item tables),
 * +16 sliding kernel off, +32 / +64 force the plane-tiled sliding plan with 4 / 8 planes per slab,
 * +128 mul_linear as the reference's composition instead of the one-pass kernel, +256 small-operand stencil kernel off,
 * +512 stencil kernel with one instead of four coefficients per thread, +1024 device-resident N-D div / exp / log
 * recurrences off (host loops of product launches), +2048 fused Horner loop of subst_var off (three launches per step),
 * +4096 axis-convolution kernel (1-d operand x N-d tensor) off, +8192 zero-extension of odd-shaped dense products to the DFMA
 * kernels' extents off, +16384 row-staged bulk-copy (TMA) variant of the Horner loop off,
 * +32768 plain small-operand products on the row-staged kernel too (slower than the gather kernel; A/B),
 * +65536 row-walking plain-load variant of the Horner loop (k_horner_direct, the default for tensors from 2^17 coefficients
 * with rows of at least 48) off, +131072 plain small-operand products with rows of at least 192 coefficients stay on the gather
 * kernel instead of k_horner_direct, +262144 plain small-operand products of any row length on k_horner_direct (A/B),
 * +524288 whole 16^3 slabs on the step-table sliding kernel instead of the run-granular k_mul_slide16 (A/B).
 * Environment (read at gtp_ctx_create): GTP_DIRECT_MIN / GTP_DIRECT_CTAS tune k_horner_direct's size threshold and CTAs per SM; GTP_LAUNCH_HIST=1 prints per-kernel launch counts and host-time shares when the
 * context is destroyed; GTP_NO_SCALAR_POOL=1 / GTP_NO_FUSED_CLS=1 switch the host-written scalar slots / the fused
 * classification off. */
int gtp_ctx_set_fast_mul(gtp_ctx* ctx, int enabled);

/* ---- multi-GPU groups (one process per GPU, SPMD; SURVEY 8e) --------------------------------- */
/* Every rank makes the same sequence of calls on replicated handles.  A group context owns one NCCL communicator on its
 * stream (NCCL is dlopen'ed: libnccl.so.2).  gtp_mul partitions a general product (:984-1012) whose result has at least
 * `threshold` coefficients (default 10^7, north_star) over the ranks by folded-cyclic leading-axis rows -- row k0 costs
 * k0 + 1 sub-products (:1001-1010), rank r owns k0 mod 2W in {r, 2W-1-r} -- and leaves the result ROW-SHARDED; the next
 * consumer that needs the whole tensor (the next product of a Horner chain :574-578, gtp_to_host, ...) replicates it with
 * one grouped NCCL broadcast per row, cached in the handle.  Everything else runs replicated. */
int gtp_nccl_unique_id(void* out128);                       /* rank 0 calls this and ships the 128 bytes to the others */
int gtp_ctx_create_group(int device, void* cuda_stream, int rank, int world, const void* id128, gtp_ctx** out);
int gtp_ctx_group_info(gtp_ctx* ctx, int* rank, int* world, uint64_t* partitioned_products, uint64_t* gathers);
int gtp_ctx_set_partition_threshold(gtp_ctx* ctx, uint64_t coefficients);   /* 0: partition every general product (tests) */
/* the row map and the block map as plain integer functions (no device needed) */
uint64_t gtp_partition_rows(uint64_t n_rows, int world, int rank, uint64_t* rows_out);
void gtp_partition_block(uint64_t n_slices, int world, int rank, uint64_t* lo, uint64_t* hi, uint64_t* block);
/* An operand uploaded in shards: `block_data` holds this rank's leading-axis slices [lo, hi) of the tensor of FULL shape
 * `shape` (gtp_partition_block); 1/W of the host-to-device traffic per rank, replicated over NVLink by one ncclAllGather
 * when first used.  gtp_from_device_block wraps a zero-padded device block of `block` slices without copying. */
int gtp_from_host_block(gtp_ctx* ctx, int ndim, const uint64_t* shape, const uint64_t* degrees_p1, const double* block_data, gtp_poly** out);
int gtp_from_device_block(gtp_ctx* ctx, int ndim, const uint64_t* shape, const uint64_t* degrees_p1, const double* device_block, gtp_poly** out);
int gtp_is_distributed(const gtp_poly* p);                  /* 1: sharded and not replicated yet */
int gtp_replicate(gtp_ctx* ctx, const gtp_poly* p);         /* collective; idempotent */
uint64_t gtp_local_rows(const gtp_poly* p, uint64_t* rows_out);   /* rows of a row-sharded result held by this rank */
int gtp_to_host_local(gtp_ctx* ctx, const gtp_poly* p, double* out); /* D2H of those rows only (no collective); synchronises */

/* ---- construction, transfer, metadata ------------------------------------------------------- */
/* TaylorPoly::new (:33-41): upload `data` (row-major over `shape`, prod(shape) doubles).  `data` may be reused or freed
 * as soon as the call returns: pageable memory is staged by the driver, and for a pinned / registered source (whose DMA
 * would run later) the call waits for the copy. */
int gtp_from_host(gtp_ctx* ctx, int ndim, const uint64_t* shape, const uint64_t* degrees_p1,
                  const double* data, gtp_poly** out);
/* Same, but wraps an existing device buffer WITHOUT copying or taking ownership (the caller keeps
 * it alive while the handle or anything cloned from it lives).  Used for NCCL-gathered operands. */
int gtp_from_device(gtp_ctx* ctx, int ndim, const uint64_t* shape, const uint64_t* degrees_p1,
                    const double* device_data, gtp_poly** out);
int gtp_to_host(gtp_ctx* ctx, const gtp_poly* p, double* out); /* into_array (:63-66); synchronises */
/* address of the stored coefficients, valid in kernels on the context's stream.  For tensors of one or two coefficients
 * created by gtp_from_scalar / gtp_var* it is a mapped pinned HOST address (unified addressing), otherwise device memory. */
int gtp_device_ptr(gtp_ctx* ctx, const gtp_poly* p, const double** out);
int gtp_clone(gtp_ctx* ctx, const gtp_poly* p, gtp_poly** out); /* Clone (:10) */
void gtp_free(gtp_ctx* ctx, gtp_poly* p);
int gtp_ndim(const gtp_poly* p);                      /* num_vars (:48-51)            */
uint64_t gtp_len(const gtp_poly* p);                  /* coeffs.len()                 */
void gtp_shape(const gtp_poly* p, uint64_t* out);     /* coeffs.shape() (stored)      */
void gtp_degrees_p1(const gtp_poly* p, uint64_t* out);/* shape() (:53-56)             */

int gtp_from_scalar(gtp_ctx* ctx, double x, gtp_poly** out);                              /* From<T> :626-630, Zero/One :638-656 */
int gtp_zero_with(gtp_ctx* ctx, int ndim, const uint64_t* degrees_p1, gtp_poly** out);     /* :208-216 */
int gtp_var(gtp_ctx* ctx, uint64_t v, double x, uint64_t len, gtp_poly** out);            /* :239-248 */
int gtp_var_at_zero(gtp_ctx* ctx, uint64_t v, uint64_t len, gtp_poly** out);              /* :228-237 */
int gtp_var_with_degrees_p1(gtp_ctx* ctx, uint64_t v, double x, int ndim, const uint64_t* degrees_p1,
                            gtp_poly** out);                                               /* :250-259 */

/* ---- operators (impl Add/Sub/Mul/Div/Neg, full reference dispatch order) --------------------- */
int gtp_add(gtp_ctx* ctx, const gtp_poly* a, const gtp_poly* b, gtp_poly** out); /* :854-882   */
int gtp_sub(gtp_ctx* ctx, const gtp_poly* a, const gtp_poly* b, gtp_poly** out); /* :911-937   */
int gtp_mul(gtp_ctx* ctx, const gtp_poly* a, const gtp_poly* b, gtp_poly** out); /* :1014-1072 */
int gtp_div(gtp_ctx* ctx, const gtp_poly* a, const gtp_poly* b, gtp_poly** out); /* :1194-1231 */
int gtp_neg(gtp_ctx* ctx, const gtp_poly* a, gtp_poly** out);                    /* :902-909   */
int gtp_exp(gtp_ctx* ctx, const gtp_poly* a, gtp_poly** out);                    /* :406-417, :1271-1317 */
int gtp_log(gtp_ctx* ctx, const gtp_poly* a, gtp_poly** out);                    /* :419-430, :1319-1386 */
int gtp_pow(gtp_ctx* ctx, const gtp_poly* a, uint32_t exp, gtp_poly** out);      /* :433-451   */

/* ---- gathers, shifts, reductions -------------------------------------------------------------- */
int gtp_derivative(gtp_ctx* ctx, const gtp_poly* a, uint64_t v, uint64_t n, gtp_poly** out);                /* :457-481 */
int gtp_taylor_expansion_of_coeff(gtp_ctx* ctx, const gtp_poly* a, uint64_t v, uint64_t n, gtp_poly** out); /* :484-509 */
int gtp_shift_down(gtp_ctx* ctx, const gtp_poly* a, uint64_t v, uint64_t n, gtp_poly** out);                /* :514-536 */
int gtp_coefficients_of_term(gtp_ctx* ctx, const gtp_poly* a, uint64_t v, uint64_t order, gtp_poly** out);  /* :341-358 */
int gtp_taylor_polynomial(gtp_ctx* ctx, const gtp_poly* a, uint64_t v, uint64_t order, gtp_poly** out);     /* :360-378 */
int gtp_taylor_polynomial_terms(gtp_ctx* ctx, const gtp_poly* a, uint64_t v, const uint64_t* orders,
                                int n_orders, gtp_poly** out);                                              /* :380-404 */
int gtp_subst_var(gtp_ctx* ctx, const gtp_poly* a, uint64_t v, const gtp_poly* subst, gtp_poly** out);      /* :540-580 */
int gtp_truncate_to_degree_p1(gtp_ctx* ctx, const gtp_poly* a, uint64_t degree_p1, gtp_poly** out);         /* :183-193 */
int gtp_remove_last_variable(gtp_ctx* ctx, const gtp_poly* a, gtp_poly** out);                              /* :172-181 */
int gtp_extend_to_dim(gtp_ctx* ctx, const gtp_poly* a, uint64_t ndim, uint64_t degree_p1, gtp_poly** out);  /* :81-89   */
/* test helper `extend` (:91-112): zero-extend the stored array to `new_size`, degrees = new_size */
int gtp_extend(gtp_ctx* ctx, const gtp_poly* a, int ndim, const uint64_t* new_size, gtp_poly** out);

/* ---- scalar readers (synchronise) ------------------------------------------------------------ */
int gtp_constant_term(gtp_ctx* ctx, const gtp_poly* a, double* out);                                  /* :296-299 */
int gtp_coefficient(gtp_ctx* ctx, const gtp_poly* a, const uint64_t* index, int n_index, double* out);/* :314-339 */
/* The callers' read-back pattern (generating_function.rs:959-965, :988-993): `count` coefficients
 * along axis v with every other index 0, as ONE gather kernel + ONE D2H copy. */
int gtp_gather_axis(gtp_ctx* ctx, const gtp_poly* a, uint64_t v, uint64_t count, double* out);
int gtp_extract_constant(gtp_ctx* ctx, const gtp_poly* a, int* is_constant, double* value);           /* :262-269 */
/* :275-294.  *is_linear = 1 and (c, m, v) filled when the polynomial is c + m*eps_v. */
int gtp_extract_linear(gtp_ctx* ctx, const gtp_poly* a, int* is_linear, double* c, double* m, uint64_t* v);
int gtp_is_zero(gtp_ctx* ctx, const gtp_poly* a, int* out);                                           /* :643-645 */
int gtp_is_one(gtp_ctx* ctx, const gtp_poly* a, int* out);                                            /* :653-655 */
int gtp_evaluate_all_one(gtp_ctx* ctx, const gtp_poly* a, double* out);                               /* :583-586 */
/* derive(PartialEq) (:10): stored shape, degrees_p1 and every coefficient (IEEE ==). */
int gtp_eq(gtp_ctx* ctx, const gtp_poly* a, const gtp_poly* b, int* out);

/* ---- the hot kernel, exposed raw for the bench and for output-axis sharding (SURVEY 8e) ------- */
/* General truncated N-D product `mul` (:984-1012), no dispatch.  Computes the leading-axis output
 * rows k0 = row_begin + i*row_step, i < row_count, of the result of shape `rshape` and writes row i
 * (prod(rshape[1:]) doubles) at out_rows + i*prod(rshape[1:]).  x, y are device buffers of shapes
 * xshape / yshape.  With row_begin = rank, row_step = world this is one rank's cyclic shard. */
int gtp_mul_rows_raw(gtp_ctx* ctx, int ndim, const uint64_t* xshape, const double* x,
                     const uint64_t* yshape, const double* y, const uint64_t* rshape,
                     uint64_t row_begin, uint64_t row_step, uint64_t row_count, double* out_rows);
/* Same for an explicit list of leading-axis rows (row rows[i] lands at out_rows + i*prod(rshape[1:])):
 * one launch for a rank's load-balanced shard, e.g. the folded-cyclic map k0 mod 2W in {r, 2W-1-r},
 * which gives every rank the same MAC count although row k0 costs (k0+1) sub-products (:1001-1010). */
int gtp_mul_rowlist_raw(gtp_ctx* ctx, int ndim, const uint64_t* xshape, const double* x,
                        const uint64_t* yshape, const double* y, const uint64_t* rshape,
                        const uint64_t* rows, uint64_t n_rows, double* out_rows);
/* MAC count of the general product (trip counts of :975-977 and :1002-1004); FLOPs = 2*MACs. */
double gtp_mul_macs(int ndim, const uint64_t* xshape, const uint64_t* yshape, const uint64_t* rshape);
/* Which kernel gtp_mul_rows_raw would pick for these shapes: 0 the bit-exact reference-order family (reference-order kernel,
 * small-operand stencil kernel, axis-convolution kernel), 2 2x2-blocked DFMA kernel, 3 sliding 1x2 DFMA kernel (dense cube
 * slabs), 6 / 7 the blocked / sliding kernel after zero-extending odd extents (27, 31, 17 ...) to supported ones. */
int gtp_mul_kernel_kind(gtp_ctx* ctx, int ndim, const uint64_t* xshape, const uint64_t* yshape,
                        const uint64_t* rshape);
/* FP64 pipe microbenchmarks (the roofline denominator): runs `iters` dependent-chain DFMA (kind 0)
 * or DMMA m8n8k4 (kind 1) per thread on a full grid and returns achieved FLOP/s in *flops. */
int gtp_fp64_peak_probe(gtp_ctx* ctx, int kind, int iters, double* flops, double* ms);

/* ---- univariate TaylorExpansion<F64> (src/univariate_taylor.rs) -------------------------------- */
int gtu_constant(gtp_ctx* ctx, double x, gtu_series** out);                           /* Constant(T) :11, From<u32> :262-266 */
int gtu_from_coefficients(gtp_ctx* ctx, const double* xs, uint64_t n, gtu_series** out); /* :62-66 */
int gtu_var(gtp_ctx* ctx, double x, uint64_t order, gtu_series** out);                /* :16-23   */
void gtu_free(gtp_ctx* ctx, gtu_series* s);
int gtu_is_constant(const gtu_series* s);
uint64_t gtu_order(const gtu_series* s);                                              /* :38-43 (GTP_UNBOUNDED for Constant) */
int gtu_to_host(gtp_ctx* ctx, const gtu_series* s, double* out);                      /* order() doubles (1 for Constant) */
int gtu_coeff(gtp_ctx* ctx, const gtu_series* s, uint64_t order, double* out);        /* :25-36   */
int gtu_derivative(gtp_ctx* ctx, const gtu_series* s, uint64_t order, double* out);   /* :45-60   */
int gtu_add(gtp_ctx* ctx, const gtu_series* a, const gtu_series* b, gtu_series** out);/* :268-306 */
int gtu_sub(gtp_ctx* ctx, const gtu_series* a, const gtu_series* b, gtu_series** out);/* :321-362 */
int gtu_mul(gtp_ctx* ctx, const gtu_series* a, const gtu_series* b, gtu_series** out);/* :364-389 */
int gtu_div(gtp_ctx* ctx, const gtu_series* a, const gtu_series* b, gtu_series** out);/* :397-439 */
int gtu_neg(gtp_ctx* ctx, const gtu_series* a, gtu_series** out);                     /* :308-319 */
int gtu_exp(gtp_ctx* ctx, const gtu_series* a, gtu_series** out);                     /* :151-168 */
int gtu_log(gtp_ctx* ctx, const gtu_series* a, gtu_series** out);                     /* :170-189 */
int gtu_pow(gtp_ctx* ctx, const gtu_series* a, uint32_t exp, gtu_series** out);       /* :192-203 */
int gtu_subst(gtp_ctx* ctx, const gtu_series* a, const gtu_series* subst, gtu_series** out); /* :93-115 */
int gtu_taylor_expansion_of_coeff(gtp_ctx* ctx, const gtu_series* a, uint64_t n, gtu_series** out); /* :69-89 */
int gtu_eq(gtp_ctx* ctx, const gtu_series* a, const gtu_series* b, int* out);         /* derive(PartialEq) :8 */

/* ---- univariate programs: a DAG of TaylorExpansion<F64> ops recorded on the host, run by one kernel launch ------------
 * Every slot is a value of the program.  Inputs (constant / var / from_coefficients) are copied at record time; an op
 * records a new slot whose variant (Constant / Polynomial) and order are known at once (gtu_program_slot).  Each op means
 * exactly the gtu_* call of the same name -- the same variant and order rules, the same errors, raised when it is
 * recorded (GTP_ERR_ARG for a bad slot or a quotient above order 2048, GTP_ERR_INDEX for GTU_MAX of a Polynomial) -- and
 * the same bits in every coefficient.  GTU_POW records the binary exponentiation of gtu_pow (`exp` is the exponent; `b`
 * is ignored, as it is for the unary ops); GTU_MAX is F64::max (x > y ? x : y) of two Constants.
 * gtu_program_run uploads the program in one host-to-device copy, runs every recorded op in one launch of a single CTA
 * (independent ops on different warps), reads the `outputs` back in one device-to-host copy and synchronises.  `out`
 * receives the outputs' coefficients one after another (1 double for a Constant, the order for a Polynomial).  A program
 * may be run again, and recorded into further between runs. */
typedef struct gtu_program gtu_program;
typedef enum gtu_op {
  GTU_ADD = 0, GTU_SUB = 1, GTU_MUL = 2, GTU_DIV = 3, GTU_NEG = 4, GTU_EXP = 5, GTU_LOG = 6, GTU_POW = 7, GTU_MAX = 8
} gtu_op;
int gtu_program_create(gtp_ctx* ctx, gtu_program** out);
void gtu_program_free(gtp_ctx* ctx, gtu_program* p);
int gtu_program_constant(gtp_ctx* ctx, gtu_program* p, double x, uint32_t* slot);
int gtu_program_var(gtp_ctx* ctx, gtu_program* p, double x, uint64_t order, uint32_t* slot);
int gtu_program_from_coefficients(gtp_ctx* ctx, gtu_program* p, const double* xs, uint64_t n, uint32_t* slot);
int gtu_program_op(gtp_ctx* ctx, gtu_program* p, int op, uint32_t a, uint32_t b, uint32_t exp, uint32_t* slot);
/* the slot's variant and order (gtu_is_constant / gtu_order: GTP_UNBOUNDED for a Constant); GTP_ERR_ARG for a bad slot */
int gtu_program_slot(const gtu_program* p, uint32_t slot, int* is_constant, uint64_t* n);
int gtu_program_run(gtp_ctx* ctx, gtu_program* p, const uint32_t* outputs, int n_outputs, double* out);

/* ---- host evaluator: an SGCL program end to end (SURVEY 8 f1) ------------------------------------ */
/* Plays the role of the reference's `genfer file.sgcl` for the default f64 Taylor mode -- run() / run_program::<F64>
 * (src/main.rs:108-227): parse (src/parser.rs), translate to a generating function (src/semantics/gf.rs), simplify
 * and evaluate it (GenFun::simplify / eval, src/generating_function.rs:474-765), moments (moments_taylor :970-1005,
 * limit 5) and probability masses (probs_taylor :937-967), post-processing and report (main.rs:301-473).  Every
 * TaylorPoly operation of that pipeline is a gtp_* call on `ctx`, i.e. runs in the CUDA library.
 *   limit  : --limit N, or -1 for the reference's automatic limit (finite support, else Markov's inequality)
 *   flags  : 1 = --no-probs, 2 = --no-simplify-gf, 4 = --bounds: run_program_intervals::<F64> (src/main.rs:145-185) -- the
 *            evaluator runs over TaylorPoly<Interval<F64>> on the device (gti_*), ratio constants are the enclosures
 *            Number::from_ratio builds (number/number.rs:26-33), the report prints "in [lo, hi]" lines (main.rs:291-299);
 *            the GenFun is evaluated unsimplified in this mode;
 *            8 = -s / --symbolic (src/main.rs:196-209, src/symbolic.rs): the generating function becomes ONE univariate
 *            computation DAG on the host (symbolic Taylor coefficients, evaluator/symbolic.hpp) and that DAG is evaluated
 *            over TaylorExpansion<F64> as a gtu_program: one launch per evaluation (the rest, the moments and the
 *            probabilities: 3 launches, 2 with --no-probs) (probs_symbolic / moments_symbolic :238-299); F64 only
 *   unroll : --unroll (reference default 8; only used by `while`)
 * On error (parse error, or anything the reference would panic on) returns GTP_ERR_INDEX and copies the message
 * into `err`.  The report is byte-compatible with the reference's stdout under --no-timing. */
typedef struct gtp_sgcl_result gtp_sgcl_result;
int gtp_run_sgcl(gtp_ctx* ctx, const char* source, int64_t limit, int flags, uint64_t unroll,
                 gtp_sgcl_result** out, char* err, size_t err_cap);
void gtp_sgcl_free(gtp_sgcl_result* r);
const char* gtp_sgcl_report(const gtp_sgcl_result* r);
/* Z, E, raw 2..4, sigma, V, central 3, central 4, skewness, kurtosis (the values the report prints) */
void gtp_sgcl_moments(const gtp_sgcl_result* r, double* out11);
uint64_t gtp_sgcl_limit(const gtp_sgcl_result* r);          /* number of probability masses computed */
int gtp_sgcl_is_normalized(const gtp_sgcl_result* r);
void gtp_sgcl_probs(const gtp_sgcl_result* r, double* unnormalized, double* normalized); /* p(i), p(i)/Z */
void gtp_sgcl_stats(const gtp_sgcl_result* r, uint64_t* nodes_evaluated, uint64_t* cache_hits);
/* the intervals behind gtp_sgcl_moments (11 lo, hi pairs) and gtp_sgcl_probs (limit pairs each; either may be null):
 * points for a plain f64 run without rest mass, the enclosures themselves for a --bounds run (flags & 4) */
void gtp_sgcl_moment_bounds(const gtp_sgcl_result* r, double* out22);
void gtp_sgcl_prob_bounds(const gtp_sgcl_result* r, double* unnormalized_pairs, double* normalized_pairs);

/* ---- Interval<F64> TaylorPoly on the device (SURVEY 8 f3) -------------------------------------------------------------
 * The number type of the reference's --bounds mode: TaylorPoly<Interval<F64>> (src/interval.rs:11-15 with the one-ulp
 * widening of :29-31 / number/f64.rs:127-171 after every operation).  `gti_poly` mirrors `gtp_poly`: each entry point
 * replaces the TaylorPoly<T> method of the same name in src/multivariate_taylor.rs at T = Interval<F64> (line numbers as
 * for the gtp_* functions above).  Coefficients cross the boundary as (lo, hi) pairs of doubles.  Products and the
 * element-wise family evaluate in the reference's term order; div / exp / log use coefficient-wise recurrences whose
 * results are valid enclosures a few ulps different from the reference's slice-wise recursion. */
typedef struct gti_poly gti_poly;
int gti_from_scalar(gtp_ctx* ctx, double lo, double hi, gti_poly** out);                                  /* :207-215 */
int gti_zero_with(gtp_ctx* ctx, int ndim, const uint64_t* degrees_p1, gti_poly** out);                    /* :66-72 */
int gti_var(gtp_ctx* ctx, uint64_t v, double lo, double hi, uint64_t len, gti_poly** out);                /* :239-248 */
int gti_var_at_zero(gtp_ctx* ctx, uint64_t v, uint64_t len, gti_poly** out);                              /* :228-237 */
int gti_var_with_degrees_p1(gtp_ctx* ctx, uint64_t v, double lo, double hi, int ndim, const uint64_t* degrees_p1,
                            gti_poly** out);                                                              /* :250-259 */
/* data: prod(shape) (lo, hi) pairs when pairs != 0, else prod(shape) doubles taken as point intervals */
int gti_from_host(gtp_ctx* ctx, int ndim, const uint64_t* shape, const uint64_t* degrees_p1, const double* data, int pairs,
                  gti_poly** out);                                                                        /* :55-64 */
int gti_to_host(gtp_ctx* ctx, const gti_poly* p, double* out_pairs);   /* 2 * gti_len(p) doubles */
void gti_free(gtp_ctx* ctx, gti_poly* p);
int gti_ndim(const gti_poly* p);
uint64_t gti_len(const gti_poly* p);
void gti_shape(const gti_poly* p, uint64_t* out);
void gti_degrees_p1(const gti_poly* p, uint64_t* out);
int gti_add(gtp_ctx* ctx, const gti_poly* a, const gti_poly* b, gti_poly** out);                          /* :854-882 */
int gti_sub(gtp_ctx* ctx, const gti_poly* a, const gti_poly* b, gti_poly** out);                          /* :911-937 */
int gti_mul(gtp_ctx* ctx, const gti_poly* a, const gti_poly* b, gti_poly** out);                          /* :1014-1072 */
int gti_div(gtp_ctx* ctx, const gti_poly* a, const gti_poly* b, gti_poly** out);                          /* :1194-1231 */
int gti_neg(gtp_ctx* ctx, const gti_poly* a, gti_poly** out);                                             /* :902-909 */
int gti_exp(gtp_ctx* ctx, const gti_poly* a, gti_poly** out);                                             /* :406-417 */
int gti_log(gtp_ctx* ctx, const gti_poly* a, gti_poly** out);                                             /* :419-430 */
int gti_pow(gtp_ctx* ctx, const gti_poly* a, uint32_t e, gti_poly** out);                                 /* :433-451 */
int gti_derivative(gtp_ctx* ctx, const gti_poly* a, uint64_t v, uint64_t n, gti_poly** out);              /* :453-483 */
int gti_taylor_expansion_of_coeff(gtp_ctx* ctx, const gti_poly* a, uint64_t v, uint64_t n, gti_poly** out); /* :485-512 */
int gti_shift_down(gtp_ctx* ctx, const gti_poly* a, uint64_t v, uint64_t n, gti_poly** out);              /* :514-536 */
int gti_coefficients_of_term(gtp_ctx* ctx, const gti_poly* a, uint64_t v, uint64_t order, gti_poly** out); /* :341-358 */
int gti_taylor_polynomial_terms(gtp_ctx* ctx, const gti_poly* a, uint64_t v, const uint64_t* orders, int n_orders,
                                gti_poly** out);                                                          /* :380-404 */
int gti_subst_var(gtp_ctx* ctx, const gti_poly* a, uint64_t v, const gti_poly* subst, gti_poly** out);    /* :538-580 */
int gti_truncate_to_degree_p1(gtp_ctx* ctx, const gti_poly* a, uint64_t degree_p1, gti_poly** out);       /* :183-193 */
int gti_remove_last_variable(gtp_ctx* ctx, const gti_poly* a, gti_poly** out);                            /* :172-181 */
int gti_extend_to_dim(gtp_ctx* ctx, const gti_poly* a, uint64_t ndim, uint64_t degree_p1, gti_poly** out); /* :81-89 */
int gti_constant_term(gtp_ctx* ctx, const gti_poly* a, double* out2);                                     /* :261-265 */
int gti_extract_constant(gtp_ctx* ctx, const gti_poly* a, int* is_constant, double* out2);                /* :217-226 */
int gti_gather_axis(gtp_ctx* ctx, const gti_poly* a, uint64_t v, uint64_t count, double* out_pairs);      /* coefficient() x count */
/* The host evaluator over gti_*: enclosures of rest mass, total mass Z, raw moments 1..4 (out12: lo, hi pairs) and of
 * the first `limit` probability masses -- the reference's `run_program::<Interval<F64>>` restricted to its direct outputs
 * (src/main.rs:150-227).  Ratio constants are the enclosures Number::from_ratio builds (number/number.rs:26-33). */
int gtp_run_sgcl_bounds(gtp_ctx* ctx, const char* source, int64_t limit, uint64_t unroll, double* out12,
                        double* probs_lohi, char* err, size_t err_cap);

#ifdef __cplusplus
}
#endif
#endif /* GENFER_TAYLOR_H */
