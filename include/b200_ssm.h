/*
 * b200_ssm.h -- C ABI of libb200ssm.so: the B200 (sm_100a) kernels behind the reference's
 * selective-scan / SS2D / SSD operator API.
 *
 * Drop-in boundary.  The reference binds its native code through the pybind11 module
 * `selective_scan_cuda` (reference CrossMamba/FusionMamba/selective_scan/selective_scan.cpp:494-497:
 * `fwd`, `bwd`), fed by the parameter blocks SSMParamsBase / SSMParamsBwd
 * (selective_scan.h:26-69, 71-101: sizes, flags, raw pointers, element strides), and calls the
 * un-vendored Triton `mamba_chunk_scan_combined` (SSD/MedSSD.py:41,361-375).  This header carries
 * the same information as plain C: no torch types, callers allocate every output, every entry
 * point is asynchronous on the given stream and returns 0 on success, <0 for an invalid argument
 * (message in b200_last_error()), >0 for a cudaError_t raised by the launch.
 *
 * Conventions: all strides are in ELEMENTS of the tensor's dtype; the sequence (last) dimension
 * of every activation tensor must have stride 1 (selective_scan.cpp:252-253,270-278).
 * Thread-safety: stateless apart from a thread-local error string; re-entrant across processes
 * (one per GPU under DDP, reference ddp_train.py:78-81).
 */
#ifndef B200_SSM_H_
#define B200_SSM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* b200_stream_t; /* cudaStream_t */

typedef enum { B200_F32 = 0, B200_BF16 = 1, B200_F16 = 2 } b200_dtype;

#define B200_SSCAN_MAX_DSTATE 16 /* this build; the reference allows 256 (selective_scan_common.h:11, MAX_DSTATE) but every model uses 16 */
#define B200_SSCAN_ROWS_PER_TASK 16

/* ------------------------------------------------------------------------------------------
 * Mamba-1 selective scan -- replaces selective_scan_cuda.fwd / .bwd
 * (selective_scan.cpp:226-336 / 338-492; kernels selective_scan_fwd_kernel.cuh:67-303,
 * selective_scan_bwd_kernel.cuh:75-489).
 *
 *   delta' = softplus?(delta + delta_bias[d])                 (x <= 20 ? log1p(exp x) : x)
 *   x_t[n] = exp(delta'_t A[d,n]) x_{t-1}[n] + delta'_t u_t B[b,g,n,t]
 *   out_t  = sum_n C[b,g,n,t] x_t[n] + D[d] u_t          (* silu(z_t) when z is given)
 *
 * Shapes: u, delta, z, out (batch, dim, L); A (dim, N) f32; B, C (batch, G, N, L) with
 * G | dim, channel d uses group d / (dim/G); D, delta_bias (dim) f32.
 *
 * Two extensions serve the SS2D cross-scan (reference MedMamba.py:393-395) without materialising
 * the four permuted copies; both default to the plain operator:
 *   - rev_mask: bit g set => group g is scanned from t = L-1 down to 0.  Inputs are read and
 *     outputs written at their memory position, so a reversed group consumes/produces tensors
 *     that are NOT flipped (torch.flip of directions 2,3 becomes free).  Requires G <= 32.
 *   - u_group_div: groups g and g' with g / u_group_div == g' / u_group_div read the same u rows
 *     (directions k and k+2 scan the same image in opposite orders).  u is then addressed as
 *       u + b*u_batch_stride + (g / u_group_div)*u_group_stride + r*u_row_stride,  r = d % (dim/G).
 *     Plain operator: u_group_div = 1, u_group_stride = (dim/G)*u_row_stride.
 *     delta (and ddelta) are addressed the same way with their own strides and no sharing:
 *       delta + b*delta_batch_stride + g*delta_group_stride + r*delta_row_stride
 *     (plain operator: delta_group_stride = (dim/G)*delta_row_stride).
 *
 * State checkpoints (replace the reference's chunk tensor `x`, selective_scan.cpp:313): the
 * forward writes the state entering every `ckpt_every`-th step into `ckpt`, laid out
 *   [task][chunk][n][16 rows, as pairs (r, r+8)] f32,  task = (b*G + g)*ceil((dim/G)/16) + row_tile,
 *   chunk = 1 .. ceil(L/ckpt_every)-1   (chunk 0 is the zero state and is never stored); opaque to callers,
 * size from b200_sscan_ckpt_bytes().  The backward recomputes inside a chunk from its checkpoint
 * (no per-step state is ever stored).  ckpt == NULL => inference, nothing written.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t batch, dim, seqlen, dstate, n_groups;
    int32_t io_dtype;       /* b200_dtype of u, delta, B, C, z, out */
    int32_t delta_softplus; /* bool */
    uint32_t rev_mask;
    int32_t u_group_div;
    int32_t ckpt_every;     /* 8; ignored when ckpt == NULL */
    int64_t u_batch_stride, u_group_stride, u_row_stride;
    int64_t delta_batch_stride, delta_group_stride, delta_row_stride; /* addressed like u (group g, row r of the group) */
    int64_t B_batch_stride, B_group_stride, B_state_stride;
    int64_t C_batch_stride, C_group_stride, C_state_stride;
    int64_t z_batch_stride, z_row_stride;
    int64_t out_batch_stride, out_row_stride;
    const void* u;
    const void* delta;
    const float* A;          /* (dim, N) contiguous */
    const void* B;
    const void* C;
    const float* D;          /* (dim) or NULL */
    const void* z;           /* or NULL */
    const float* delta_bias; /* (dim) or NULL */
    void* out;               /* (batch, dim, L) io_dtype; gated by silu(z) when z != NULL */
    float* last_state;       /* (batch, dim, N) contiguous f32, or NULL */
    float* ckpt;             /* see above, or NULL */
} b200_sscan_fwd_params;

typedef struct {
    b200_sscan_fwd_params f; /* same inputs as the forward; f.out / f.last_state unused; f.ckpt required */
    /* dout is addressed like u: dout + b*dout_batch_stride + (g / dout_group_div)*dout_group_stride
       + r*dout_row_stride, so that the two directions that receive the same upstream gradient
       (cross-merge adjoint) share one tensor.  Plain operator: dout_group_div = 1,
       dout_group_stride = (dim/G)*dout_row_stride. */
    int64_t dout_batch_stride, dout_group_stride, dout_row_stride;
    int64_t dout_group_div;
    int64_t du_batch_stride, du_row_stride;
    int64_t ddelta_batch_stride, ddelta_group_stride, ddelta_row_stride;
    int64_t dB_batch_stride, dB_group_stride, dB_state_stride;
    int64_t dC_batch_stride, dC_group_stride, dC_state_stride;
    int64_t dz_batch_stride, dz_row_stride;
    const void* dout; /* (batch, dim, L) io_dtype */
    void* du;         /* (batch, dim, L) io_dtype: one row per (b, d) even when u rows are shared */
    void* ddelta;     /* (batch, dim, L) io_dtype */
    void* dz;         /* (batch, dim, L) io_dtype, required iff f.z != NULL */
    /* The next five are ACCUMULATED with fp32 atomics (like selective_scan.cpp:460-466):
       the caller zero-fills them first.  dB/dC are (batch, G, N, L) f32 whatever io_dtype is
       (selective_scan.cpp:461-462), rows of L contiguous, addressed through their strides (contiguous:
       G*N*L, N*L, L) -- like delta / ddelta they may live inside a wider buffer (SS2D keeps B, C, delta of all
       four directions in ONE projection output and their gradients in one buffer of the same layout). */
    float* dA;          /* (dim, N) */
    float* dB;
    float* dC;
    float* dD;          /* (dim) or NULL */
    float* ddelta_bias; /* (dim) or NULL */
} b200_sscan_bwd_params;

size_t b200_sscan_ckpt_bytes(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate,
                             int32_t n_groups, int32_t ckpt_every);
int b200_sscan_fwd(const b200_sscan_fwd_params* p, b200_stream_t stream);
int b200_sscan_bwd(const b200_sscan_bwd_params* p, b200_stream_t stream);
/* Which kernel the calling thread's last b200_sscan_fwd / _bwd launched:
 *   1 = sscan.cu (every layout sscan2.cu cannot take: L % 4 != 0, unaligned views, 16-bit I/O, the z gate in the backward),
 *   2 = the TMA-staged kernels of sscan2.cu (fp32 tensors whose layouts tensor maps can describe: L % 4 == 0, 16-byte aligned
 *       bases and strides),
 *   3 = sscan.cu with its opt-in TMA row staging (B200_SSCAN_TMA=1, fp32 with tensor-map-describable u / delta / dout).
 * Both generations share the checkpoint format; for profilers and tests. */
int b200_sscan_last_variant(void);

/* ------------------------------------------------------------------------------------------
 * Strided twins of the cross-scan pack for the fused SS2D core (medical_image_classification_b200/cross.py::SS2DCoreFn;
 * reference MedMamba.py:393-400): x2 is addressed as x2 + b*batch_stride + i*layout_stride + d*row_stride (i = 0 row-major
 * plane, 1 column-major plane; rows of L contiguous), so that it can live in the (2, D, B, L) layout in which the x_proj /
 * dt_proj contraction is one GEMM over B*L columns.  b200_cross_scan_unpack4 is the whole adjoint in one pass:
 * dx (B, D, H, W) = du[b,0,d] + du[b,1,d] + gx2[b,0,d] + (du[b,2,d] + du[b,3,d] + gx2[b,1,d])^T with du (B, 4, D, L) contiguous
 * (the scan's du per direction: hw, hw reversed, wh, wh reversed, all at memory positions) and gx2 laid out like x2.  f32.
 * ------------------------------------------------------------------------------------------ */
int b200_cross_scan_pack_strided(const float* x, float* x2, int64_t x2_batch_stride, int64_t x2_layout_stride, int64_t x2_row_stride,
                                 int32_t batch, int32_t D, int32_t H, int32_t W, b200_stream_t stream);
int b200_cross_scan_unpack4(const float* du, const float* gx2, int64_t x2_batch_stride, int64_t x2_layout_stride, int64_t x2_row_stride,
                            float* dx, int32_t batch, int32_t D, int32_t H, int32_t W, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * EfficientVMamba atrous scan / merge, step 2 (SURVEY.md 8(f) rank 4) -- replaces EfficientScan / EfficientMerge of
 * CrossMamba/FusionMamba/models/cross.py:139-190 / 34-92 (strided slices, transposes and four copies each way).
 *   scan : x (B, C, H, W) -> xs (B, 4, C, H2*W2), H2 = ceil(H/2), W2 = ceil(W/2):
 *          xs[b,k,c,idx] = x[b, c, 2i + (k&1), 2j + (k>>1)], idx = i*W2 + j for k even, j*H2 + i for k odd; zero beyond the image
 *   merge: ys (B, 4, C, H2*W2) -> y (B, C, H, W), the inverse scatter.  Each is the other's adjoint (autograd uses that).
 *   dtype in {F32, BF16, F16}; (H + 1) * (W + 2) <= 8192.
 * ------------------------------------------------------------------------------------------ */
int b200_atrous_scan(const void* x, void* xs, int32_t batch, int32_t C, int32_t H, int32_t W, int32_t dtype, b200_stream_t stream);
int b200_atrous_merge(const void* ys, void* y, int32_t batch, int32_t C, int32_t H, int32_t W, int32_t dtype, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * SS2D cross-scan / cross-merge helpers (reference MedMamba.py:393-395, 420-424, 476-477).
 *
 * b200_cross_scan_pack:  x (batch, D, H, W)  ->  x2 (batch, 2, D, L):  x2[:,0] = x row-major,
 *   x2[:,1] = x transposed (column-major order).  With rev_mask = 0b1100 and u_group_div = 1 on a
 *   direction order (hw, wh, hw-reversed, wh-reversed) this is all the data movement the four
 *   directions need.
 * b200_cross_merge:  ys (batch, 4, D, L) as written by the scan with rev_mask (every direction at
 *   its memory position)  ->  y (batch, L, D) = ys0 + ys2 + transpose(ys1 + ys3), i.e. the sum of
 *   the four un-permuted directions laid out (B, H, W, D).
 * b200_cross_merge_bwd: dy (batch, L, D) -> dys2 (batch, 2, D, L) (the adjoint scatter): [0] feeds
 *   directions 0 and 1, [1] (column-major planes) feeds directions 2 and 3 (dout_group_div = 2).
 * ------------------------------------------------------------------------------------------ */
int b200_cross_scan_pack(const void* x, void* x2, int32_t batch, int32_t D, int32_t H, int32_t W,
                         int32_t dtype, b200_stream_t stream);
int b200_cross_scan_pack_bwd(const void* dx2, void* dx, int32_t batch, int32_t D, int32_t H, int32_t W,
                             int32_t dtype, b200_stream_t stream);
int b200_cross_merge(const void* ys, void* y, int32_t batch, int32_t D, int32_t H, int32_t W,
                     int32_t dtype, b200_stream_t stream);
int b200_cross_merge_bwd(const void* dy, void* dys, int32_t batch, int32_t D, int32_t H, int32_t W,
                         int32_t dtype, b200_stream_t stream);

/* SSD twin of the cross-scan / cross-merge (reference SSD/MedSSD.py:332-336, 376-391; CrossMamba_fusion_2b2.py:280-289,
 * 344-356).  The Mamba-2 operator mixes the four directions' B / C inside one state group, so the four orderings are
 * materialised, in one pass each way:
 *   b200_cross_scan4: x (batch, C, H, W) f32 planes with batch stride x_batch_stride (a channel slice of a wider
 *     tensor is read in place) -> x4 (batch, 4, C, L): k=0 row-major, k=1 column-major, k=2 / k=3 their reversals.
 *   b200_cross_scan4_bwd: dx4 -> dx (the four un-permuted gradients added up).
 *   b200_ssd_merge4: y (batch, L, 4, d) f32 (the SSD output with direction-major heads) -> out (batch, L, d) =
 *     y[l,0] + y[L-1-l,2] + y[lT,1] + y[L-1-lT,3], lT = w H + h;   b200_ssd_merge4_bwd: dout -> dy (a gather). */
int b200_cross_scan4(const float* x, int64_t x_batch_stride, float* x4, int32_t batch, int32_t C, int32_t H, int32_t W,
                     b200_stream_t stream);
int b200_cross_scan4_bwd(const float* dx4, float* dx, int64_t dx_batch_stride, int32_t batch, int32_t C, int32_t H, int32_t W,
                         b200_stream_t stream);
int b200_ssd_merge4(const float* y, float* out, int32_t batch, int32_t d, int32_t H, int32_t W, b200_stream_t stream);
int b200_ssd_merge4_bwd(const float* dout, float* dy, int32_t batch, int32_t d, int32_t H, int32_t W, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Mamba-2 SSD -- replaces mamba_ssm.ops.triton.ssd_combined.mamba_chunk_scan_combined
 * (call contract: reference SSD/MedSSD.py:344-375).
 *
 *   dt'   = clamp(softplus?(dt + dt_bias[h]), dt_min, dt_max)
 *   S_t   = exp(dt'_t A[h]) S_{t-1} + dt'_t x_t (outer) B_t        S: (P, N) per (batch, head)
 *   y_t   = S_t C_t + D[h] x_t                                    (* silu(z_t) when z is given)
 *
 * x, out (batch, L, H, P); dt (batch, L, H); B, C (batch, L, G, N); A, D, dt_bias (H) f32.
 * Every tensor is addressed by explicit element strides (the reference passes permuted views
 * whose L stride is 1, SURVEY.md section 3.3).  The gate z, D with a head dimension, seq_idx and
 * cu_seqlens are never passed by the reference models (SSD/MedSSD.py:361-375) and are rejected
 * by the host wrapper.  Evaluated chunk-wise (chunk_size steps): Y = (C B^T o decay) (dt X) +
 * decay C S_prev, S_c = decay S_{c-1} + B^T (decay dt X); all contractions on tensor cores.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t batch, seqlen, nheads, headdim, n_groups, dstate, chunk_size;
    int32_t io_dtype;   /* x, dt, B, C, out */
    int32_t dt_softplus;
    int32_t precision;  /* 0: fp32-accurate tensor-core products (3xTF32 split); 1: single-pass TF32
                           (what the reference's Triton kernels do on fp32 inputs; exact for bf16 data) */
    float dt_min, dt_max;
    int64_t x_stride[4];   /* batch, L, head, p */
    int64_t dt_stride[3];  /* batch, L, head */
    int64_t B_stride[4];   /* batch, L, group, n */
    int64_t C_stride[4];
    int64_t out_stride[4];
    const void* x;
    const void* dt;
    const float* A;        /* (H) */
    const void* B;
    const void* C;
    const float* D;        /* (H) or NULL */
    const float* dt_bias;  /* (H) or NULL */
    const float* initial_states; /* (batch, H, P, N) contiguous f32 or NULL */
    void* out;             /* (batch, L, H, P) io_dtype */
    float* final_states;   /* (batch, H, P, N) contiguous f32 or NULL */
    float* workspace;      /* b200_ssd_workspace_bytes() bytes, kept for the backward:
                              dt' [b][h][c][Q] | cumsum(dt' A) [b][h][c][Q] | chunk-entry states
                              [b][c][h][P][N] | C B^T [b][c][g][Q][Q] */
} b200_ssd_fwd_params;

typedef struct {
    b200_ssd_fwd_params f;  /* forward inputs + its workspace (f.out / f.final_states unused) */
    int64_t dout_stride[4];
    const void* dout;
    /* gradients: fp32 in the logical shapes of their primals (strides below), written (not accumulated)
       except the three reduced over batch/sequence, which the caller zero-fills */
    float* dx;       /* (batch, L, H, P) */
    float* ddt;      /* (batch, L, H) */
    float* dB;       /* (batch, L, G, N) */
    float* dC;       /* (batch, L, G, N) */
    float* dA;       /* (H)   accumulated */
    float* dD;       /* (H) or NULL, accumulated */
    float* ddt_bias; /* (H) or NULL, accumulated */
    float* scratch;  /* b200_ssd_bwd_scratch_bytes() bytes */
    /* element strides of dx (batch, L, head, p), ddt (batch, L, head), dB / dC (batch, L, group, n).  All zero = contiguous in
       the logical shape.  The models pass the strides of the primals (sequence-contiguous views, SSD/MedSSD.py:344-347), so the
       gradients come back in the layout the cross-scan adjoint reads and no strided copy follows. */
    int64_t dx_stride[4];
    int64_t ddt_stride[3];
    int64_t dB_stride[4];
    int64_t dC_stride[4];
} b200_ssd_bwd_params;

size_t b200_ssd_workspace_bytes(int32_t batch, int32_t seqlen, int32_t nheads, int32_t headdim,
                                int32_t n_groups, int32_t dstate, int32_t chunk_size);
size_t b200_ssd_bwd_scratch_bytes(int32_t batch, int32_t seqlen, int32_t nheads, int32_t headdim,
                                  int32_t n_groups, int32_t dstate, int32_t chunk_size);
int b200_ssd_fwd(const b200_ssd_fwd_params* p, b200_stream_t stream);
int b200_ssd_bwd(const b200_ssd_bwd_params* p, b200_stream_t stream);

/* Gated RMSNorm used by SS2D_with_SSD (reference SSD/MedSSD.py:268-269,393-394;
 * mamba_ssm.ops.triton.layernorm_gated.RMSNorm with norm_before_gate=False, one group):
 *   y = rmsnorm(x * silu(z)) * w,   rows of length `dim`, fp32.  rstd (rows) is kept for backward. */
int b200_rmsnorm_gated_fwd(const float* x, const float* z, const float* w, float* y, float* rstd,
                           int64_t rows, int32_t dim, float eps, b200_stream_t stream);
int b200_rmsnorm_gated_bwd(const float* x, const float* z, const float* w, const float* rstd,
                           const float* dy, float* dx, float* dz, float* dw_partial /* (grid, dim) */,
                           int32_t dw_rows, int64_t rows, int32_t dim, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Gated RMSNorm with groups: every configuration of mamba_ssm's layernorm_gated RMSNorm / rmsnorm_fn (mamba_ssm 2.2.2,
 * rms_norm_ref), which SS2D_with_SSD builds as RMSNorm(d_ssm, norm_before_gate, group_size = d_ssm / ngroups) (reference
 * SSD/MedSSD.py:268-269, 393-394).  Rows of `dim` columns, cut into dim / group_size contiguous groups normalised on their own:
 *   norm_before_gate = 0:  out = rmsnorm_g(x * silu(z)) * w [+ b]
 *   norm_before_gate = 1:  out = (rmsnorm_g(x) * w [+ b]) * silu(z)
 *   z == NULL:             out = rmsnorm_g(x) * w [+ b],          rmsnorm_g(v) = v * rsqrt(mean over the group of v^2 + eps)
 * All arithmetic in fp32.  x, z (rows, dim) in {F32, BF16, F16}, each with its own dtype and row stride in elements, read in place
 * (z may be a column slice of in_proj's output with any pitch); w (dim) f32; b (dim) f32 or NULL; out (rows, dim) contiguous
 * out_dtype in {F32, BF16, F16}; rstd (rows, dim / group_size) f32, kept for the backward.
 * Backward: dy (rows, dim) dy_dtype with row stride dy_row_stride -> dx (rows, dim) x_dtype and dz (rows, dim) z_dtype, contiguous
 * (dz given exactly when z is); dw_partial, db_partial (b200_rmsnorm_grid(rows, dim, group_size), dim) f32 per-CTA partial sums,
 * which the caller adds up (no atomics: reproducible); db_partial may be NULL.
 * group_size must divide dim, dim <= 8192.  Anything else returns < 0 with a message (b200_rmsnorm_grid too).
 * ------------------------------------------------------------------------------------------ */
int b200_rmsnorm_grid(int64_t rows, int32_t dim, int32_t group_size);
int b200_rmsnorm_fwd(const void* x, int32_t x_dtype, int64_t x_row_stride, const void* z, int32_t z_dtype, int64_t z_row_stride,
                     const float* w, const float* b, void* out, int32_t out_dtype, float* rstd, int64_t rows, int32_t dim,
                     int32_t group_size, int32_t norm_before_gate, float eps, b200_stream_t stream);
int b200_rmsnorm_bwd(const void* dy, int32_t dy_dtype, int64_t dy_row_stride, const void* x, int32_t x_dtype, int64_t x_row_stride,
                     const void* z, int32_t z_dtype, int64_t z_row_stride, const float* w, const float* b, const float* rstd,
                     void* dx, void* dz, float* dw_partial, float* db_partial, int64_t rows, int32_t dim, int32_t group_size,
                     int32_t norm_before_gate, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * SS2D output stage (SURVEY.md 8(f) rank 1): out = LayerNorm(y) * silu(z) and its backward -- replaces
 * `y = self.out_norm(y); y = y * F.silu(z)` (reference MedMamba.py:478-479; nn.LayerNorm(d_inner), eps 1e-5)
 * and the four autograd kernels behind it.
 *   z == NULL (and dz == NULL) gives the plain LayerNorm of the block's pre-norm (MedMamba.py:531 `self.ln_1`).
 *   y (rows, D) y_dtype in {F32, BF16} with row stride y_row_stride (the cross-merge output, or the right half of the
 *   block input read in place; BF16 -- the residual stream of an autocast model after PatchMerging's Linear -- only with
 *   z == NULL); z (rows, D) with row stride z_row_stride (the second
 *   half of in_proj's output, read in place), z_dtype in {F32, BF16}; w, b (D) f32; out (rows, D) out_dtype
 *   in {F32, BF16 (= what the following Linear would cast to under autocast)}; mean, rstd (rows) f32 kept for
 *   the backward.  Backward: dout (rows, D) out_dtype -> dy (rows, D) y_dtype, dz (rows, D) z_dtype contiguous,
 *   dw_partial / db_partial (b200_ln_gate_grid(rows), D) f32 per-CTA partial sums (the caller adds the rows up).
 *   D <= 1024.
 * ------------------------------------------------------------------------------------------ */
int b200_ln_gate_grid(int64_t rows);
int b200_ln_gate_fwd(const void* y, int32_t y_dtype, int64_t y_row_stride, const void* z, int64_t z_row_stride, int32_t z_dtype,
                     const float* w, const float* b, void* out, int32_t out_dtype, float* mean, float* rstd, int64_t rows, int32_t D,
                     float eps, b200_stream_t stream);
int b200_ln_gate_bwd(const void* dout, const void* y, int32_t y_dtype, int64_t y_row_stride, const void* z, int64_t z_row_stride,
                     int32_t z_dtype, const float* w, const float* b, int32_t out_dtype, const float* mean, const float* rstd, void* dy,
                     void* dz, float* dw_partial, float* db_partial, int64_t rows, int32_t D, b200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * SS2D producer stage (SURVEY.md 8(f) rank 1): x = SiLU(depthwise conv3x3(x_in) + bias) -- replaces
 * `x.permute(0,3,1,2).contiguous()`, `self.act(self.conv2d(x))` (reference MedMamba.py:470-473; Conv2d(D, D, 3,
 * padding=1, groups=D)) and the `.float()` before the scan (MedMamba.py:403).
 *   xin: channels-last (B, H, W, D) view, element (b,h,w,d) at ((b*H + h)*W + w)*pix_stride + d (the x half of
 *   in_proj's output, pix_stride = 2 D), in_dtype in {F32, BF16}; weight (D, 3, 3) f32; bias (D) f32 or NULL;
 *   out (B, D, H, W) f32 planes (what b200_cross_scan_pack reads).  W <= 64.
 *   Backward: gout (B, D, H, W) f32 -> dxin (B, H, W, D) contiguous in_dtype; dweight (D, 9), dbias (D) f32 are
 *   ACCUMULATED with atomics (the caller zero-fills them); dbias may be NULL.
 * ------------------------------------------------------------------------------------------ */
int b200_dwconv_silu_fwd(const void* xin, int64_t pix_stride, int32_t in_dtype, const float* weight, const float* bias, float* out,
                         int32_t B, int32_t D, int32_t H, int32_t W, b200_stream_t stream);
int b200_dwconv_silu_bwd(const float* gout, const void* xin, int64_t pix_stride, int32_t in_dtype, const float* weight,
                         const float* bias, void* dxin, float* dweight, float* dbias, int32_t B, int32_t D, int32_t H, int32_t W,
                         b200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Block tail (SURVEY.md 8(f) rank 2): out = channel_shuffle(cat(left, x), groups = 2) + input -- replaces the
 * permute / cat / shuffle copy / residual add of SS_Conv_SSM.forward (reference MedMamba.py:486-499, 533-538).
 *   left (B, c, P) planes, or (B, P, c) when left_channels_last (the conv branch run in torch.channels_last; P = H*W),
 *   and x (B, P, c) channels-last (the SS2D branch), both lx_dtype
 *   in {F32, BF16}; input, out (B, P, 2 c) io_dtype: F32, or BF16 with BF16 left / x (the residual stream of an autocast
 *   model is bf16 after PatchMerging's Linear; the sum is formed in fp32 and rounded once, as torch does).
 *   out[b,p,2j] = left[b,j,p] + input[b,p,2j]; out[b,p,2j+1] = x[b,p,j] + input[b,p,2j+1].
 *   Backward: dout (B, P, 2 c) io_dtype -> dleft (B, c, P), dx (B, P, c) in lx_dtype (the gradient of `input` is dout).
 * ------------------------------------------------------------------------------------------ */
int b200_shuffle_cat_add_fwd(const void* left, int32_t left_channels_last, const void* x, int32_t lx_dtype, const void* input,
                             void* out, int32_t io_dtype, int32_t B, int32_t c, int32_t P, b200_stream_t stream);
int b200_shuffle_cat_add_bwd(const void* dout, int32_t io_dtype, void* dleft, int32_t left_channels_last, void* dx, int32_t lx_dtype,
                             int32_t B, int32_t c, int32_t P, b200_stream_t stream);

/* PatchMerging2D gather (reference MedMamba.py:186-204, `x0..x3 = x[:, i::2, j::2, :]`, `torch.cat`): x (batch, H, W, C) ->
 * out (batch, H/2, W/2, 4 C), out[b, h2, w2, k C + c] = x[b, 2 h2 + (k & 1), 2 w2 + (k >> 1), c]; pixel_bytes = C * element size,
 * a multiple of 16.  inverse != 0: the adjoint, x = d out (batch, H/2, W/2, 4 C) -> out = d x (batch, H, W, C). */
int b200_patch_merge(const void* x, void* out, int32_t batch, int32_t H, int32_t W, int32_t pixel_bytes, int32_t inverse,
                     b200_stream_t stream);

/* ------------------------------------------------------------------------------------------ */
const char* b200_last_error(void);   /* thread-local message of the last failing call */
int b200_version(void);              /* ABI version, bumped on any struct change */
int b200_kernel_launches(void);      /* number of kernels this library has launched in this process */
size_t b200_sizeof_params(int32_t which); /* 0 sscan_fwd, 1 sscan_bwd, 2 ssd_fwd, 3 ssd_bwd: lets a binding check its struct layout */

#ifdef __cplusplus
}
#endif
#endif /* B200_SSM_H_ */
