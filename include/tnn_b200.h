/*
 * tnn_b200.h -- C ABI of libtnn_b200.so, the B200 (sm_100a) execution engine behind
 * tinynn-autograd's forward/backward tensor ops.
 *
 * The reference (borgwang/tinynn-autograd) has no FFI: its seam is the Python module API of
 * core/tensor.py and core/ops.py, whose bodies are numpy calls.  Every entry point below
 * replaces one family of those numpy call sites; the reference file:line each one stands in
 * for is cited next to it.  The host side (core/_backend.py) binds these with ctypes.
 *
 * Conventions
 *   - plain pointers and sizes only; every device pointer comes from tnn_alloc()
 *   - every call returns 0 on success, non-zero on failure; tnn_last_error() describes it
 *   - one process = one device = one compute stream; calls are asynchronous w.r.t. the GPU
 *     except tnn_d2h / tnn_sync / tnn_event_elapsed_ms
 *   - dtype: TNN_F32 = 0, TNN_F64 = 1 (reference tensors are float32 params / float64 tests)
 *   - shapes/strides are int64 element counts, rank <= TNN_MAX_DIMS, row-major;
 *     a stride of 0 means "broadcast along this axis" (numpy broadcasting, ops.py:32-213)
 */
#ifndef TNN_B200_H
#define TNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TNN_MAX_DIMS 8
#define TNN_F32 0
#define TNN_F64 1

/* ---- elementwise op codes (tnn_ew) ------------------------------------------------------ */
enum {
  /* binary: out = f(x, y) */
  TNN_OP_ADD = 0,      /* ops.py:33   add_ forward                                  */
  TNN_OP_SUB = 1,      /* ops.py:61   sub_ (= add(neg)) fused                        */
  TNN_OP_MUL = 2,      /* ops.py:66   mul_ forward; ops.py:72,81 grad*other          */
  TNN_OP_DIV = 3,      /* ops.py:94   div_ forward; ops.py:100 grad/ts2              */
  TNN_OP_POW = 4,      /* ops.py:122  pow_ forward                                   */
  TNN_OP_MAXIMUM = 5,  /* ops.py:167  np.maximum                                     */
  TNN_OP_MINIMUM = 6,  /* ops.py:192  np.minimum                                     */
  TNN_OP_GE = 7,       /* tensor.py:54 __ge__  (1.0 / 0.0 in dtype)                  */
  TNN_OP_GT = 8,       /* tensor.py:48 __gt__                                        */
  TNN_OP_LE = 9,       /* tensor.py:57 __le__                                        */
  TNN_OP_LT = 10,      /* tensor.py:51 __lt__                                        */
  TNN_OP_EQ = 11,
  /* ternary: out = f(x, y, z), x is the incoming gradient */
  TNN_OP_MUL_GE = 20,     /* x*(y>=z)   ops.py:170 maximum_ grad ts1                 */
  TNN_OP_MUL_GT = 21,     /* x*(y> z)   ops.py:179 maximum_ grad ts2                 */
  TNN_OP_MUL_LE = 22,     /* x*(y<=z)   ops.py:195 minimum_ grad ts1                 */
  TNN_OP_MUL_LT = 23,     /* x*(y< z)   ops.py:204 minimum_ grad ts2                 */
  TNN_OP_MUL_EQ = 24,     /* x*(y==z)   ops.py:229,238 max_/min_ grad                */
  TNN_OP_DIV_BWD_B = 25,  /* -x*y/(z*z) ops.py:109 div_ grad ts2 (y=ts1, z=ts2)      */
  TNN_OP_POW_BWD_A = 26,  /* x*z*y**(z-1)    ops.py:128 pow_ grad ts1                */
  TNN_OP_POW_BWD_B = 27,  /* x*(log(y)*z)    ops.py:138 pow_ grad ts2 (z = y**b)     */
  /* unary: out = f(x) (p0, p1 are scalar parameters) */
  TNN_OP_NEG = 40,        /* ops.py:294 neg_                                          */
  TNN_OP_EXP = 41,        /* ops.py:217 exp_                                          */
  TNN_OP_LOG = 42,        /* ops.py:244 log_                                          */
  TNN_OP_COPY = 43,
  TNN_OP_CLIP = 44,       /* ops.py:334 x.clip(p0,p1); flags bit0 = has min, bit1 = has max */
  TNN_OP_SCALE = 45,      /* x*p0 + p1                                                */
  TNN_OP_CLIP_BWD = 46,   /* binary: x*(mask(y; p0,p1))  ops.py:336-343               */
  TNN_OP_RECIP_MUL = 47,  /* binary: x / y -- alias of DIV kept for log_ grad ops.py:247 */
  /* activations (core/layers.py LeakyReLU, ELU, GELU, Softplus, SiLU; new).  Unary forward
     y = f(x), p0 = slope / alpha:
       LEAKY_RELU  x if x >= 0 else p0 x                     f' = 1 if x >= 0 else p0
       ELU         x if x >= 0 else p0 expm1(x)              f' = 1 if x >= 0 else p0 exp(x)
       GELU        x Phi(x), Phi(x) = erfc(-x/sqrt2)/2       f' = Phi(x) + x phi(x),
                                                                  phi(x) = exp(-x^2/2)/sqrt(2 pi)
       GELU_TANH   x s, s = sigma(2u) (= (1 + tanh u)/2),    f' = s + 2x s(1-s) sqrt(2/pi)(1 + 0.134145 x^2)
                   u = sqrt(2/pi)(x + 0.044715 x^3)
       SOFTPLUS    max(x, 0) + log1p(exp(-|x|))              f' = sigma(x)
       SILU        x sigma(x)                                f' = sigma(x)(1 + x(1 - sigma(x)))
     sigma(v) = 1/(1+e^-v) for v >= 0, e^v/(1+e^v) otherwise; s(1-s) is evaluated as sigma(v) sigma(-v).
     The kink at 0 goes to the x >= 0 branch (ReLU's convention: LeakyReLU(0) is ReLU on non-NaN x).
     NaN gives NaN in y and in dx; +-inf give the function's limit and the derivative's limit; every
     finite x gives a finite y and dx (terms whose weight underflowed to 0 are 0, never inf * 0).
     Computed in the operands' dtype with libdevice's accurate functions (no fast-math); Phi is
     libdevice's normcdf, and GELU_TANH evaluates no tanh. */
  TNN_OP_LEAKY_RELU = 48,
  TNN_OP_ELU = 49,
  TNN_OP_GELU = 50,
  TNN_OP_GELU_TANH = 51,
  TNN_OP_SOFTPLUS = 52,
  TNN_OP_SILU = 53,
  /* binary backward: out = x * f'(y), x = the upstream gradient, y = the activation's input, p0 as
     the forward's (laid out as TNN_OP_CLIP_BWD) */
  TNN_OP_LEAKY_RELU_BWD = 60,
  TNN_OP_ELU_BWD = 61,
  TNN_OP_GELU_BWD = 62,
  TNN_OP_GELU_TANH_BWD = 63,
  TNN_OP_SOFTPLUS_BWD = 64,
  TNN_OP_SILU_BWD = 65
};

/* ---- reduction op codes (tnn_reduce) ------------------------------------------------------ */
enum { TNN_RED_SUM = 0, TNN_RED_MAX = 1, TNN_RED_MIN = 2 };

/* ---- optimizer codes (tnn_opt_step), core/optimizer.py ------------------------------------ */
enum {
  TNN_OPT_SGD = 0,      /* optimizer.py:46  */
  TNN_OPT_ADAM = 1,     /* optimizer.py:67  */
  TNN_OPT_RMSPROP = 2,  /* optimizer.py:107 */
  TNN_OPT_MOMENTUM = 3, /* optimizer.py:126 */
  TNN_OPT_ADAGRAD = 4,  /* optimizer.py:143 */
  TNN_OPT_ADADELTA = 5, /* optimizer.py:158 */
  TNN_OPT_ADAMW = 6,    /* decoupled weight decay (Loshchilov & Hutter) */
  TNN_OPT_RADAM = 7,    /* rectified Adam (Liu et al.) */
  TNN_OPT_ADAMAX = 8    /* Adam's infinity-norm variant (Kingma & Ba, section 7) */
};

/* ---- lifecycle / errors ------------------------------------------------------------------- */
const char* tnn_last_error(void);
int tnn_init(int device);                 /* selects the device, creates the compute + copy streams */
int tnn_shutdown(void);
int tnn_sync(void);                       /* cudaStreamSynchronize(compute stream) */
int tnn_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem, size_t* l2_bytes);
int tnn_device_count(int* n);
void* tnn_stream(void);                   /* the cudaStream_t every kernel is launched on */
uint64_t tnn_launch_count(void);          /* number of kernels this library has launched   */

/* ---- memory: stream-ordered caching pool (replaces numpy's implicit malloc) ---------------- */
int tnn_alloc(size_t nbytes, void** out);
void* tnn_alloc_ptr(size_t nbytes);       /* same, returns the pointer; NULL on failure */
int tnn_free(void* p);
int tnn_pool_stats(size_t* reserved_bytes, size_t* in_use_bytes, size_t* n_cuda_malloc);
int tnn_pool_trim(void);
int tnn_h2d(void* dst, const void* src, size_t nbytes);  /* src reusable on return */
int tnn_d2h(void* dst, const void* src, size_t nbytes);  /* blocks until the bytes are on the host */
/* Asynchronous read-back: copies `nbytes` of `src` into PINNED host memory on a dedicated stream,
 * ordered after the compute work queued so far but not after anything queued later, and records
 * `done_event` (tnn_event_create) when the bytes have landed; tnn_event_sync makes the host wait for
 * it.  Lets a training loop log step i's loss (run.py:84 `loss.values`) while step i+1 is queued. */
int tnn_d2h_async(void* pinned_dst, const void* src, size_t nbytes, void* done_event);
int tnn_event_sync(void* ev);
int tnn_d2d(void* dst, const void* src, size_t nbytes);
int tnn_memset(void* dst, int byte, size_t nbytes);
int tnn_host_alloc(size_t nbytes, void** out);            /* pinned host memory */
int tnn_host_free(void* p);
int tnn_host_register(void* p, size_t nbytes);            /* pin caller-owned host memory in place */
int tnn_host_unregister(void* p);
/* copy-stream plumbing for input prefetch (run.py:78 batches overlap the previous step) */
int tnn_h2d_async_copy_stream(void* dst, const void* pinned_src, size_t nbytes);
int tnn_copy_stream_sync(void);           /* host waits until queued copies are done (staging reuse) */
int tnn_copy_wait_compute(void);          /* copy stream waits for work queued so far on compute */
int tnn_compute_wait_copy(void);          /* compute stream waits for copies queued so far       */
/* events on the compute stream (bench timing) */
int tnn_event_create(void** ev);
int tnn_event_destroy(void* ev);
int tnn_event_record(void* ev);
int tnn_event_elapsed_ms(void* start, void* stop, float* ms); /* synchronises on stop */
/* per-kernel-family profiling: brackets every launch of `family` with events */
int tnn_prof_enable(int family);          /* 0 = off, 1 = tcgen05 GEMM, 2 = SIMT GEMM, 3 = tf32 split */
int tnn_prof_collect(double* total_ms, uint64_t* n_launches); /* synchronises, then resets */
int tnn_l2_flush(void);                   /* writes a buffer larger than L2 */

/* ---- captured steps (CUDA graphs) -----------------------------------------------------------
 * One training step of examples/mnist/run.py:78-83 (zero_grad, forward, loss, backward, step) is
 * ~35 launches of a few microseconds each; issued one at a time from Python it is launch-bound.
 * Everything queued on the compute stream between tnn_graph_begin and tnn_graph_end (kernels,
 * memsets, device copies, NCCL collectives) is recorded instead of executed; tnn_graph_launch
 * replays it with one call.  Blocks handed out by tnn_alloc during the capture belong to the
 * graph (addresses are baked into its nodes): they are reused inside the capture but only return
 * to the pool at tnn_graph_destroy.  tnn_h2d / tnn_d2h fail during a capture. */
int tnn_graph_begin(void);
int tnn_graph_end(void** graph_out);
int tnn_graph_abort(void);                /* drop a capture in progress (host-side error path) */
int tnn_graph_launch(void* graph);        /* one replay on the compute stream */
int tnn_graph_info(void* graph, size_t* n_nodes, size_t* n_kernel_nodes, size_t* n_blocks);
int tnn_graph_destroy(void* graph);

/* ---- elementwise with numpy broadcasting (core/ops.py:32-249, 293-299, 333-344) ------------ */
/* out is contiguous with shape[ndim]; xs/ys/zs are element strides (0 = broadcast); y, z may be
 * NULL for unary/binary ops. p0/p1/flags are op parameters (clip bounds, scale). */
int tnn_ew(int op, int dtype, void* out, const void* x, const void* y, const void* z,
           int ndim, const int64_t* shape,
           const int64_t* xs, const int64_t* ys, const int64_t* zs,
           double p0, double p1, int flags);
/* fast path: every operand is contiguous with n elements, or a single element (mask bit set) */
int tnn_ew_flat(int op, int dtype, void* out, const void* x, const void* y, const void* z,
                int64_t n, int scalar_mask, double p0, double p1, int flags);
int tnn_cast(int dst_dtype, void* dst, int src_dtype, const void* src, int64_t n);
int tnn_fill(int dtype, void* dst, double value, int64_t n);

/* ---- reductions (ops.py:225-265) and the un-broadcast sum (ops.py:41-46 and 11 copies) ----- */
/* x viewed as (outer, red, inner) contiguous; out has (outer, inner) */
int tnn_reduce(int red_op, int dtype, void* out, const void* x,
               int64_t outer, int64_t red, int64_t inner);
/* grad (gshape[ndim], contiguous) summed over every axis where keep[i]==0 -> out contiguous */
int tnn_unbroadcast(int dtype, void* out, const void* grad, int ndim,
                    const int64_t* gshape, const int32_t* keep);

/* ---- layout (ops.py:268-330) --------------------------------------------------------------- */
/* generic strided copy: dst[doff + sum i_k*ds_k] = src[soff + sum i_k*ss_k], i in shape */
int tnn_strided_copy(int dtype, void* dst, const void* src, int ndim, const int64_t* shape,
                     const int64_t* dst_strides, const int64_t* src_strides);
/* getitem_ with an int64 row-index vector (data_iterator.py:27-28): out[i,:] = x[idx[i],:] */
int tnn_gather_rows(int dtype, void* out, const void* x, const int64_t* idx_dev,
                    int64_t n_idx, int64_t row_elems, int64_t n_rows_src);
/* getitem_ backward, assignment semantics (ops.py:285-288): out[idx[i],:] = g[i,:] */
int tnn_scatter_rows(int dtype, void* out, const void* g, const int64_t* idx_dev,
                     int64_t n_idx, int64_t row_elems, int64_t n_rows_dst);
/* arbitrary numpy key, flattened: out[i] = x[flat_idx[i]] / out[flat_idx[i]] = g[i] */
int tnn_gather_flat(int dtype, void* out, const void* x, const int64_t* idx_dev, int64_t n);
int tnn_scatter_flat(int dtype, void* out, const void* g, const int64_t* idx_dev, int64_t n);
/* dense one-hot label rows built on the device from int32 class labels: the `np.eye(C)[targets]`
 * of examples/mnist/run.py:27-28 (get_one_hot) without shipping B*C floats over PCIe.
 * out[r, c] = (labels[r] == c), out is (B, C) contiguous in `dtype` */
int tnn_one_hot(int dtype, void* out, const int32_t* labels_dev, int64_t B, int64_t C);

/* ---- GEMM (ops.py:150-163 dot_: A@B, grad@B.T, A.T@grad) ----------------------------------- */
/* SIMT path, any shape, f32/f64.  C[M,N] (ldc) = op(A)[M,K] * op(B)[K,N] (+ bias[N]) (+ C).
 * A(i,k) = A[i*a_rs + k*a_cs], B(k,j) = B[k*b_rs + j*b_cs]; flags bit0 = accumulate into C.
 * act_out (may be NULL, pitch ldc) additionally receives ReLU(C): Dense + ReLU in one launch; with
 * mask_src (pitch ldc) it receives C * (mask_src >= 0) instead: the dX product and the ReLU
 * backward of the layer below (ops.py:156-157 + 342-343) in one launch.
 * Products with few 32x32 tiles and K >= 128 run as a thread-block cluster along K (partials are
 * folded in rank order over distributed shared memory: deterministic, no scratch). */
int tnn_gemm_simt(int dtype, void* C, int64_t ldc, const void* A, int64_t a_rs, int64_t a_cs,
                  const void* B, int64_t b_rs, int64_t b_cs, int64_t M, int64_t N, int64_t K,
                  const void* bias, int flags, void* act_out, const void* mask_src);
/* The three gradient products of a SMALL Dense layer (ops.py:156-160 and the bias un-broadcast
 * ops.py:49-55) in one grouped SIMT launch: dx[B,K] = g[B,N] @ w[K,N]^T (dx may be NULL: the first
 * layer's input needs no gradient), dx_masked[B,K] = dx * (mask_src >= 0) (may be NULL; the ReLU
 * backward of the layer below), dw[K,N] (+)= x[B,K]^T @ g, db[1,N] (+)= column sums of g.  All
 * arrays contiguous row-major.  Meant for layers whose products are a handful of 32x32 tiles (the
 * examples/mnist MLP), where a launch costs more than the arithmetic. */
int tnn_dense_bwd_simt(int dtype, const void* g, const void* x, const void* w, const void* mask_src,
                       void* dx, void* dx_masked, void* dw, int dw_accumulate, void* db,
                       int db_accumulate, int64_t B, int64_t K, int64_t N);
/* fp32 -> (hi, lo) tf32 planes for the 3xTF32 tensor-core GEMM.  x is [R, C] row-major (ld = C).
 * plain planes  hi/lo  : [R, ldp]  (ldp >= C, multiple of 4)   -- may be NULL
 * transposed    hiT/loT: [C, ldt]  (ldt >= R, multiple of 4)   -- may be NULL */
int tnn_split_tf32(const float* x, int64_t R, int64_t C,
                   float* hi, float* lo, int64_t ldp, float* hiT, float* loT, int64_t ldt);
/* tcgen05 3xTF32: D[M,N] (ldd) = A[M,K] * B[K,N] from tf32 hi/lo planes.
 * layout bit0 = 0: A planes are K-major, stored [M, lda] (k contiguous);  1: MN-major, stored [K, lda]
 * layout bit1 = 0: B planes are K-major, stored [N, ldb] (k contiguous);  2: MN-major, stored [K, ldb]
 * so X@W is layout 2, G@W.T is layout 0 and X.T@G is layout 3, all on un-transposed planes.
 * flags bit0 = accumulate into D, bit1 = relu on the output; bias[N] may be NULL.
 * Fused activation outputs (Dense -> ReLU -> next Dense without extra passes, layers.py:49,97-98):
 * act_out (may be NULL, pitch ldd) receives ReLU(D) while D keeps the pre-activation the ReLU
 * backward mask needs; act_hi/act_lo (may be NULL, pitch ld_act) receive the tf32 planes of
 * ReLU(D), i.e. the A operand of the next layer's product.  act_out may be NULL while the planes
 * are given: the fp32 ReLU output is then not written at all (nothing in a training step reads it).
 * Backward form: with mask_src (pitch ldd) set, act_out = D * (mask_src >= 0) instead -- the dX
 * product of a layer whose input came out of a ReLU hands back both dL/da (D) and dL/dz (act_out,
 * with tf32 planes for the dW / dX products it feeds), ops.py:342-343 fused into ops.py:156-157. */
int tnn_gemm_tf32x3(float* D, int64_t ldd,
                    const float* a_hi, const float* a_lo, int64_t lda,
                    const float* b_hi, const float* b_lo, int64_t ldb,
                    int64_t M, int64_t N, int64_t K, const float* bias, int flags, int layout,
                    float* act_out, float* act_hi, float* act_lo, int64_t ld_act,
                    const float* mask_src);
/* Mixed split (default path): the two cross terms of the 3xTF32 expansion need only ~9 significant
 * bits per factor, so they run as BF16 MMAs at twice the TF32 rate:
 *     A*B ~= bf16(A - A_hi)*bf16(B) + bf16(A)*bf16(B - B_hi) + A_hi*B_hi,   A_hi = tf32(A)
 * 8 tensor-pipe slots per 32-wide K block instead of 12, same 8 B/element of planes.  Split error
 * 7e-7 of max|A@B| (3xTF32: 7e-8), below the fp32 accumulation error of the K loop.
 * tnn_split_tf32_bf16: x [R, C] -> hi (fp32 plane, tf32 values), h16 = bf16(x), l16 = bf16(x - hi),
 *   all with pitch ld elements (multiple of 8, >= C; pad columns are zeroed).
 * tnn_gemm_tf32_bf16x2: same contract as tnn_gemm_tf32x3 (layout bits, flags, fused activation
 *   outputs, mask_src), operands and the activation planes in the three-plane form. */
int tnn_split_tf32_bf16(const float* x, int64_t R, int64_t C, float* hi, void* h16, void* l16,
                        int64_t ld);
int tnn_gemm_tf32_bf16x2(float* D, int64_t ldd,
                         const float* a_hi, const void* a_h16, const void* a_l16, int64_t lda,
                         const float* b_hi, const void* b_h16, const void* b_l16, int64_t ldb,
                         int64_t M, int64_t N, int64_t K, const float* bias, int flags, int layout,
                         float* act_out, float* act_hi, void* act_h16, void* act_l16, int64_t ld_act,
                         const float* mask_src);
/* Scaled two-plane split (the default path since r02): the 3xTF32 expansion with every factor in 16
 * bits.  X = x * 2^e (one e per tensor: max|X| in [2^14, 2^15)), hf = fp16(X) (the mantissa tf32
 * keeps), l = fp16(X - hf);
 *     A*B ~= 2^-(ea+eb) * ( l_A*hf_B + hf_A*l_B + hf_A*hf_B )
 * as three tcgen05 kind::f16 MMAs per K=16 step on 4 B/element of planes.  Element error
 * <= 2^-20 * max(|x|, 2^-19 max|x_tensor|); replaces ops.py:150-160 `@`.
 * Each operand carries a 32-byte device record `meta` {u32 bits of max|x|, u32 statistics-missing
 * flag, i32 e, i32 safe, u32 small-element count, u32 non-zero count, u32 ticket, u32 pad}:
 * tnn_f16_stats      zeroes the record and fills max|x| (relu_mode: of relu(x)).
 * tnn_f16_meta_reset zeroes a record a producer kernel is about to fill (tnn_gemm_f16x3 stat_meta).
 * tnn_split_f16      derives e from max|x|, writes the planes (pitch ld, multiple of 8, pad columns
 *                    zeroed) and, from what it counts while writing, `safe`: the tensor is finite and at
 *                    most 1/256 of its non-zero elements lie below 2^-5 after scaling (the level under
 *                    which the residual plane goes subnormal).
 * tnn_gemm_f16x3     layout bits / flags 1, 2 as tnn_gemm_tf32x3; returns at once ON THE DEVICE
 *                    unless both operands are safe.  act_out (optional) = relu(D), or with mask_src
 *                    D * (mask_src >= 0) (ops.py:336-343 fused into the dX product).  stat_meta
 *                    (optional): statistics of the result -- of act_out's values when act_out or
 *                    mask_src is given, of relu(D) with flags & 8 -- for the split of the next product.
 * tnn_split_tf32_bf16_cond / tnn_gemm_tf32_bf16x2_cond: the fallback for operands outside the guard,
 *   launched unconditionally behind tnn_gemm_f16x3: they return at once when both records say safe,
 *   otherwise split (relu_mode: relu(x)) / multiply with the mixed split above.  No host round trip.
 *   The split takes both operands in one launch.  result_meta (optional): the record tnn_gemm_f16x3
 *   would have filled with its result's statistics; the fallback marks it "statistics missing" and
 * tnn_f16_stats_cond, launched before the next split of that result, then computes them (it returns
 *   at once otherwise). */
int tnn_f16_stats(const float* x, int64_t n, void* meta, int relu_mode);
/* cluster shape of tnn_gemm_f16x3: 2 = one CTA pair per tile (default); 4 = two pairs on adjacent tile
 * columns sharing their A rows by TMA multicast (fewer operand bytes, but only 33 such clusters are
 * co-resident on B200: measured slower, kept as an option; also TNN_F16_CLUSTER). */
int tnn_set_gemm_f16_cluster(int cl);
int tnn_f16_meta_reset(void* meta);
int tnn_split_f16(const float* x, int64_t R, int64_t C, void* hf, void* l16, int64_t ld, void* meta,
                  int relu_mode);
int tnn_gemm_f16x3(float* D, int64_t ldd, const void* a_hf, const void* a_l16, int64_t lda,
                   const void* a_meta, const void* b_hf, const void* b_l16, int64_t ldb,
                   const void* b_meta, int64_t M, int64_t N, int64_t K, const float* bias, int flags,
                   int layout, float* act_out, const float* mask_src, void* stat_meta);
int tnn_split_tf32_bf16_cond(const float* xa, int64_t Ra, int64_t Ca, float* hia, void* h16a, void* l16a,
                             int64_t lda, int relu_a, const float* xb, int64_t Rb, int64_t Cb, float* hib,
                             void* h16b, void* l16b, int64_t ldb, int relu_b, const void* meta_a,
                             const void* meta_b, void* result_meta);
int tnn_f16_stats_cond(const float* x, int64_t n, void* meta, int relu_mode);
int tnn_gemm_tf32_bf16x2_cond(float* D, int64_t ldd, const float* a_hi, const void* a_h16,
                              const void* a_l16, int64_t lda, const float* b_hi, const void* b_h16,
                              const void* b_l16, int64_t ldb, int64_t M, int64_t N, int64_t K,
                              const float* bias, int flags, int layout, float* act_out,
                              const float* mask_src, const void* meta_a, const void* meta_b);
/* CTA-group size of the tcgen05 kernel: 1 = one CTA per SM (tile 128x256), 2 = CTA pair with
 * cta_group::2 (tile 256x256), 0 = library default.  Also settable with TNN_GEMM_CG. */
int tnn_set_gemm_cta_group(int cg);
/* The persistent tcgen05 grid leaves `n` SMs unoccupied (0..64, default 0): room for a collective
 * kernel on another stream to run beside the backward pass (the per-layer gradient all-reduce of
 * core/_dist.py).  Also settable with TNN_GEMM_RESERVED_SMS. */
int tnn_set_gemm_reserved_sms(int n);
/* Ordered split-K of the tcgen05 kernel: 0 = automatic (only the tiles of a ragged last wave are
 * cut along K, e.g. the 4096x4096x8192 dW products: 256 tiles on 74 CTA pairs), 1 = off, 2 / 4 =
 * every tile.  The K ranges of a tile are added in a fixed order, so results are deterministic.
 * Also TNN_GEMM_KSPLIT. */
int tnn_set_gemm_ksplit(int ks);
/* Tile rasterisation of the tcgen05 kernel: consecutive tiles walk `gm` tile-rows before moving
 * to the next tile column (1 = row-major order). */
int tnn_set_gemm_group_m(int gm);

/* ---- fused layer ops ----------------------------------------------------------------------- */
/* ReLU = clip(x, 0.0) (layers.py:97-98); backward mask is x >= 0 (ops.py:336-343) */
int tnn_relu_fwd(int dtype, void* out, const void* x, int64_t n);
int tnn_relu_bwd(int dtype, void* dx, const void* g, const void* x, int64_t n);
/* column sum of a (R, C) gradient = bias gradient (ops.py:49-55 on the (1,N) bias) */
int tnn_colsum(int dtype, void* out, const void* g, int64_t R, int64_t C);

/* ---- convolution / pooling passes, NHWC (new: no reference counterpart) ---------------------
 * Conv2D is im2col + the GEMM route above (core/layers.py); MaxPool2D is one pass each way.
 * x is (N, H, W, C) contiguous; the window is (KH, KW) (pooling: (PH, PW)), the stride (SH, SW),
 * PH0 / PW0 the padding before the first row / column, (OH, OW) the output extent.  One launch
 * each, no atomics (the backward passes gather in a fixed order: bit-reproducible), no host sync.
 * tnn_im2col: col[(n,oh,ow), (kh,kw,c)] = x[n, oh*SH+kh-PH0, ow*SW+kw-PW0, c], 0 in the padding;
 *   col is (N*OH*OW, KH*KW*C) row-major, so col @ w.reshape(KH*KW*C, C_out) is the convolution.
 * tnn_col2im: its adjoint, dx (N, H, W, C) WRITTEN (not accumulated): each element sums the dcol
 *   entries that read it, in ascending (kh, kw) order. */
int tnn_im2col(int dtype, void* col, const void* x, int64_t N, int64_t H, int64_t W, int64_t C,
               int64_t KH, int64_t KW, int64_t SH, int64_t SW, int64_t PH0, int64_t PW0,
               int64_t OH, int64_t OW);
int tnn_col2im(int dtype, void* dx, const void* dcol, int64_t N, int64_t H, int64_t W, int64_t C,
               int64_t KH, int64_t KW, int64_t SH, int64_t SW, int64_t PH0, int64_t PW0,
               int64_t OH, int64_t OW);
/* tnn_maxpool_fwd: y (N, OH, OW, C) = max over the real (unpadded) elements of each window, and
 *   arg (same shape, int32) = the selected element's offset INSIDE its window, kh*PW + kw: the first
 *   maximum in row-major window order, or the first NaN (np.max / np.argmax of the window).
 * tnn_maxpool_bwd: dx (N, H, W, C) WRITTEN: each element sums dy over the windows that cover it and
 *   whose arg points at it (overlapping windows included). */
int tnn_maxpool_fwd(int dtype, void* y, int32_t* arg, const void* x, int64_t N, int64_t H, int64_t W,
                    int64_t C, int64_t PH, int64_t PW, int64_t SH, int64_t SW, int64_t PH0, int64_t PW0,
                    int64_t OH, int64_t OW);
int tnn_maxpool_bwd(int dtype, void* dx, const void* dy, const int32_t* arg, int64_t N, int64_t H,
                    int64_t W, int64_t C, int64_t PH, int64_t PW, int64_t SH, int64_t SW, int64_t PH0,
                    int64_t PW0, int64_t OH, int64_t OW);

/* ---- batch normalisation over the rows of an (M, C) matrix (new: no reference counterpart) --
 * BatchNormalization in core/layers.py; x, y, dy, dx are (M, C) contiguous in `dtype`, gamma, beta
 * and the running statistics are C values of the same dtype.  mr is 2C + 1 float64 values: the
 * column means, r = 1/sqrt(var + eps) and the row count M the statistics were taken over (global
 * under data parallelism).  Statistics and sums are float64; no atomics on values, no host sync.
 * tnn_bn_stats: TRAIN statistics (biased variance) of x.  part == NULL: writes mr and updates the
 *   running statistics in place, running = (1 - momentum) * running + momentum * batch value, the
 *   variance unbiased (* M / (M - 1)); M >= 2.  part != NULL: writes the local (M, mean[C], M2[C])
 *   to part (1 + 2C float64) instead and touches nothing else.
 * tnn_bn_merge: `world` such parts (gathered in rank order) -> mr and the running update as above,
 *   merged in rank order (every rank computes the same bits). */
int tnn_bn_stats(int dtype, const void* x, int64_t M, int64_t C, double momentum, double eps, void* running_mean,
                 void* running_var, double* mr, double* part);
int tnn_bn_merge(int dtype, const double* gathered, int world, int64_t C, double momentum, double eps,
                 void* running_mean, void* running_var, double* mr);
/* tnn_bn_apply: y = (x - mean) * r * gamma + beta.  running_mean == NULL: mean and r from mr (TRAIN);
 *   otherwise from the running statistics (TEST), and they are written to mr for backward. */
int tnn_bn_apply(int dtype, void* y, const void* x, int64_t M, int64_t C, const void* gamma, const void* beta,
                 double* mr, const void* running_mean, const void* running_var, double eps);
/* tnn_bn_bwd_reduce: sums = (sum_rows dy, sum_rows dy * xhat), 2C float64, xhat = (x - mean) * r
 *   recomputed from mr; dbeta = the first C, dgamma = the second, each WRITTEN or (acc_* != 0) added
 *   to what it holds; a NULL dgamma / dbeta is skipped.
 * tnn_bn_dx: dx = gamma * r * (dy - sums[c] / M - xhat * sums[C + c] / M), M = mr[2C] (TRAIN), or
 *   dx = gamma * r * dy when sums == NULL (TEST: the statistics are constants). */
int tnn_bn_bwd_reduce(int dtype, const void* dy, const void* x, int64_t M, int64_t C, const double* mr,
                      double* sums, void* dgamma, int acc_gamma, void* dbeta, int acc_beta);
int tnn_bn_dx(int dtype, void* dx, const void* dy, const void* x, int64_t M, int64_t C, const double* mr,
              const void* gamma, const double* sums);

/* ---- pointwise losses (new: no reference counterpart) ------------------------------------------
 * MSELoss, MAELoss, HuberLoss and SigmoidCrossEntropyLoss in core/losses.py:
 *   L = (1/m_global) * sum over the n elements of l(p, t),  e = p - t,  `kind`:
 *   TNN_LOSS_MSE         l = e^2                                            dl/dp = 2e
 *   TNN_LOSS_MAE         l = |e|                                            dl/dp = sign(e), 0 at e = 0
 *   TNN_LOSS_HUBER       l = e^2/2 if |e| < delta, else delta(|e| - delta/2)   dl/dp = e, else delta sign(e)
 *   TNN_LOSS_SIGMOID_CE  p are logits z, t targets in [0, 1]:
 *                        l = max(z, 0) - z t + log1p(exp(-|z|))             dl/dz = sigmoid(z) - t
 * p, t and dp are n contiguous values of `dtype` (TNN_F32 / TNN_F64); n may be 0.  m_global >= 1 is
 * the row count of the global batch (data parallel: local rows * world).  delta (Huber only) is
 * finite and > 0.  Terms, derivatives and sums are float64, each result rounded once to dtype; the
 * sum is folded in a fixed order (no atomics on values, no host sync), so the bits do not change
 * from run to run.
 * tnn_pointwise_loss: loss_dev[0] = L, one launch.  dp (optional, else NULL) receives dL/dp for the
 *   upstream gradient 1 (the seed of loss.backward()) in the same pass, bit-identical to
 *   tnn_pointwise_loss_bwd with g = 1.
 * tnn_pointwise_loss_bwd: dp = dl/dp * (g / m_global), g = g_dev[0] (dtype, on the device); the seeded
 *   output is dl/dp * (1 / m_global). */
enum { TNN_LOSS_MSE = 0, TNN_LOSS_MAE = 1, TNN_LOSS_HUBER = 2, TNN_LOSS_SIGMOID_CE = 3 };
int tnn_pointwise_loss(int dtype, int kind, const void* p, const void* t, int64_t n, double m_global,
                       double delta, void* loss_dev, void* dp);
int tnn_pointwise_loss_bwd(int dtype, int kind, void* dp, const void* p, const void* t, int64_t n,
                           double m_global, double delta, const void* g_dev);

/* SoftmaxCrossEntropyLoss.loss (losses.py:24-32) with its batch-GLOBAL max and normaliser.
 * Stage 1: local max + local sum exp(z - local max) -> stats_dev[0..1] (device, dtype of z).
 * (data parallel: all-gather stats across ranks, merge on host or with tnn_ce_merge_stats)
 * Stage 2: given global (M, S) in stats_dev[0..1] and m = global batch:
 *          q_i = sum_j exp(z_ij-M)/S * y_ij, loss_partial = -(1/m) sum_i ln q_i -> loss_dev[0]
 * Backward: dz = gscale * (exp(z-M)/S - (1/m) y*exp(z-M)/(S q_i)), gscale read from g_dev[0]. */
int tnn_ce_stats(int dtype, const void* z, int64_t B, int64_t C, void* stats_dev);
int tnn_ce_merge_stats(int dtype, void* stats_out_dev, const void* stats_all_dev, int n_ranks);
/* labels_dev (optional, tnn_ce_loss and tnn_ce_bwd): the targets as B int32 class indices instead of
 * the dense one-hot rows y (then y may be NULL): q_i = p_{i,label_i}, the one non-zero term of the sum
 * over the one-hot row -- bit-identical results without reading B x C labels (run.py:27-28 builds
 * the dense rows with get_one_hot; utils/data_iterator.PrefetchIterator ships the indices). */
int tnn_ce_loss(int dtype, const void* z, int y_dtype, const void* y, int64_t B, int64_t C,
                const void* stats_dev, double m_global, void* q_dev, void* loss_dev,
                const int32_t* labels_dev);
/* stages 1 + 2 in ONE single-CTA launch for small logits (B <= 2048, B*C <= 16384: the
 * examples/mnist 128 x 10 case), single process only; same arithmetic and order as the staged path */
int tnn_ce_fwd_small(int dtype, const void* z, int y_dtype, const void* y, int64_t B, int64_t C,
                     double m_global, void* stats_dev, void* q_dev, void* loss_dev,
                     void* dz_dev /* optional [B,C]: dL/dz for the upstream gradient 1 (the seed of
                                     loss.backward(), tensor.py:160), bit-identical to tnn_ce_bwd with
                                     g = 1 -- the step's backward pass then skips that launch */);
int tnn_ce_bwd(int dtype, void* dz, const void* z, int y_dtype, const void* y, int64_t B, int64_t C,
               const void* stats_dev, const void* q_dev, double m_global, const void* g_dev,
               void* stat_meta /* optional, float32: a zeroed f16 operand record (tnn_f16_meta_reset)
                                  that receives max|dz| for the next tnn_split_f16 */,
               const int32_t* labels_dev);

/* Small-MLP tail in ONE launch (examples/mnist/run.py:59-84 at batch 128: layers 2..L of the
 * 784-200-100-70-30-10 network).  Phase 1, 4 batch rows per CTA with the tail's weights resident in
 * shared memory: forward of the tail Dense/ReLU layers (layers.py:43-49, 97-98), the global-softmax
 * cross-entropy (losses.py:24-32; one grid-wide exchange of (max, sum-exp) pairs), dL/dz and the dX
 * chain with ReLU masks (ops.py:156-157, 336-343).  Phase 2, after a grid-wide rendezvous: the tail's
 * dW / db (ops.py:159-160, 49-55) as 32x32 tiles over all batch rows, each element summed by one
 * thread in row order (deterministic), written straight into `grad`.
 *   in_dims/out_dims[n_layers]  widths of the tail layers (each <= 256, chained); batch <= 256
 *   w[l] [in,out], b[l] [out]   float32 parameters
 *   grad_off[2*l], [2*l+1]      element offsets of dW_l, db_l relative to `grad` (the first tail
 *                               parameter's slot of the flat gradient arena; n_grad bounds them)
 *   z1 [B,in[0]]                pre-activation of the layer BELOW the tail (its ReLU is applied here)
 *   y [B,out[L-1]]              labels, y_dtype TNN_F32 or TNN_F64;  m_global = batch size in the loss
 *   dz1 [B,in[0]]               receives dL/dz1 (masked): input of the first layer's own backward launch
 *   workspace                   scratch [scratch_floats], stats [2*n_ctas], loss_part [n_ctas],
 *                               counters [16 x uint32, zeroed once]; sizes from tnn_mlp_tail_workspace */
int tnn_mlp_tail_workspace(int n_layers, const int64_t* in_dims, const int64_t* out_dims, int64_t batch,
                           int64_t* smem_bytes, int64_t* n_ctas, int64_t* scratch_floats);
int tnn_mlp_tail_step(int n_layers, const int64_t* in_dims, const int64_t* out_dims, const void* const* w,
                      const void* const* b, const int64_t* grad_off, void* grad, int64_t n_grad,
                      const void* z1, const void* y, int y_dtype, int64_t B, double m_global, void* dz1,
                      void* loss_out, void* scratch, void* stats, void* loss_part, void* counters,
                      void* logits_out /* optional [B,out[L-1]] float32: the network's output rows
                                          (model.py:27-28 forward's return value) */);

/* fused optimizer step on flat buffers (optimizer.py:12-35 flatten + _compute_step + model.py:59-61
 * param += step).  s0/s1 are the optimizer state vectors (Adam m,v; RMSProp ms,mom; ...), h[] the
 * hyper-parameters:
 *   SGD [lr]; ADAM [lr, b1, b2, eps, 1-b1^t, 1-b2^t]; RMSPROP [lr, decay, momentum, eps];
 *   MOMENTUM [lr, momentum]; ADAGRAD [lr, eps]; ADADELTA [lr, decay, eps];
 *   ADAMW [lr, b1, b2, eps, 1-b1^t, 1-b2^t, 1-lr*wd]: Adam's step, then param = param*h[6] + step
 *     (with param NULL, step_out receives Adam's step alone and the caller adds the decay);
 *   RADAM [lr, b1, b2, eps, 1-b1^t, sqrt(1-b2^t), r_t]: mh = m/h[4]; step = -lr*r_t*mh*h[5]/(sqrt(v)+eps)
 *     if r_t > 0, else -lr*mh.  r_t is the rectification term, 0 while rho_t <= 5; the kernel reads it
 *     at run time, so a recorded step switches branch when the uploaded r_t becomes positive;
 *   ADAMAX [lr, b1, b2, eps, lr/(1-b1^t)]: u = max(b2*u, |g|+eps) (NaN propagates); step = -h[4]*m/u.
 *   every rule: h[7] = weight-decay coefficient, 0 = off (optimizer.py:28-29 `_step -= wd * v`,
 *   commented out upstream and therefore opt-in here; needs param != NULL).  AdamW passes 0 there.
 * param (updated in place: param += step) and step_out (receives step) may each be NULL. */
int tnn_opt_step(int opt, int dtype, void* param, void* step_out, const void* grad, void* s0,
                 void* s1, int64_t n, const double* h, int n_h);
/* same, with the 8 hyper-parameter doubles read from DEVICE memory at run time: the form a
 * captured step uses, because Adam's 1-b^t terms (optimizer.py:74-75) change at every replay */
int tnn_opt_step_dev(int opt, int dtype, void* param, void* step_out, const void* grad, void* s0,
                     void* s1, int64_t n, const double* h_dev);

/* ---- data-parallel collectives (new: the reference has none; SURVEY 8e) -------------------- */
int tnn_nccl_unique_id(void* id128);                       /* 128-byte ncclUniqueId */
int tnn_nccl_init(int rank, int world, const void* id128);
int tnn_nccl_destroy(void);
int tnn_allreduce_sum(int dtype, void* buf, int64_t n);    /* in place, compute stream */
int tnn_allgather(int dtype, void* recv, const void* send, int64_t n_per_rank);
/* chunked all-reduce on a second (comm) stream, so the optimiser kernel of chunk i runs while chunk
 * i+1 is on the wire: tnn_comm_wait_compute(); { tnn_allreduce_sum_comm(chunk); tnn_compute_wait_comm();
 * tnn_opt_step(chunk) } per chunk */
int tnn_comm_wait_compute(void);          /* comm stream waits for work queued so far on compute   */
int tnn_compute_wait_comm(void);          /* compute stream waits for collectives queued so far    */
int tnn_allreduce_sum_comm(int dtype, void* buf, int64_t n);   /* in place, comm stream           */
int tnn_nccl_version(int* v);

#ifdef __cplusplus
}
#endif
#endif /* TNN_B200_H */
