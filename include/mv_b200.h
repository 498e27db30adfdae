/*
 * mv_b200.h — C ABI of the B200-native (sm_100a) hot path of myrtle-vision's quantised ViT
 * training step.  Plain pointers and sizes only; no torch types.  Every entry point
 *   - works on caller-owned device buffers (no allocation inside),
 *   - is ordered on the CUDA stream passed as the last argument (a cudaStream_t cast to void*),
 *   - never synchronises the host,
 *   - returns 0 on success, non-zero on error with the message in mv_last_error().
 *
 * Reference interfaces replaced (paths relative to the myrtle-vision repository):
 *   B2, the fake-quant operator boundary:
 *     src/myrtle_vision/utils/quantize.py:47-72  qtorch.quant.Quantizer(FloatingPoint|FixedPoint..)
 *     src/myrtle_vision/utils/quantize.py:84     quant(X.data.float())  -> quant_cuda.float_quantize_nearest(a, man, exp)
 *     QPyTorch 0.3.0 pybind surface (third-party, setup.py:10): float_quantize_{nearest,stochastic},
 *     fixed_point_quantize_{nearest,stochastic}[_mask], block_quantize_{nearest,stochastic}
 *   the torch/ATen ops under ViT.forward (src/myrtle_vision/models/vit.py:267-320):
 *     torch.nn.qat.Linear.forward  (F.linear(x, weight_fake_quant(W), b) + activation_post_process)
 *     nn.LayerNorm (:37), nn.GELU (:49), Attention.forward (:84-99), Residual.forward (:26-27)
 *   and their autograd backward (straight-through quantisers, utils/quantize.py:87-89).
 */
#ifndef MV_B200_H
#define MV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* element container types */
#define MV_F32 0
#define MV_F16 1

/* rounding modes (qtorch: "nearest" / "stochastic") */
#define MV_ROUND_NEAREST 0
#define MV_ROUND_STOCHASTIC 1

const char* mv_last_error(void);
int mv_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int64_t mv_launch_count(void);

/* ---------------------------------------------------------------- fake-quant (B2)
 * qtorch.quant.float_quantize(x, exp, man, rounding)   [quant_cuda.float_quantize_*]
 * in: fp32 [n]; out: container out_dtype [n] (MV_F32, or MV_F16 when the format fits fp16:
 * exp<=5, man<=10).  Stochastic rounding adds random bits to the 23 - man bits that are dropped.
 *   man >= 7 (at most 16 bits dropped — every format the reference configures): the "16-bit stream": element i uses
 *     half-word (i&7) of Philox4x32-10(key=seed, counter={i>>3, offset}) — the low half of word (i&7)>>1 for even i,
 *     the high half for odd i — so that one Philox call serves eight elements (mv_philox_bits16 dumps it);
 *   man <  7: the "32-bit stream": word (i&3) of Philox4x32-10(key=seed, counter={i>>2, offset}) (mv_philox_bits).
 * in == out is allowed for MV_F32. */
int mv_float_quantize(const float* in, void* out, int out_dtype, int64_t n, int exp_bits,
                      int man_bits, int rounding, uint64_t seed, uint64_t offset, void* stream);

/* qtorch.quant.fixed_point_quantize(x, wl, fl, clamp, symmetric, rounding)
 * mask (nullable): uint8 [n], 1 where the value was clamped (the *_mask variants; they always
 * clamp).  Stochastic: r = (philox word >> 8) * 2^-24 in [0,1). */
int mv_fixed_point_quantize(const float* in, float* out, uint8_t* mask, int64_t n, int wl, int fl,
                            int clamp, int symmetric, int rounding, uint64_t seed,
                            uint64_t offset, void* stream);

/* qtorch.quant.block_quantize(x, wl, dim, rounding).  The tensor is viewed as
 * [outer, dsize, inner] with `dim` the middle axis; whole_tensor != 0 means dim = -1 (one block).
 * workspace: max(dsize,1) floats of scratch.  Stochastic rounding draws its tail bits like mv_float_quantize with
 * man = wl: the 16-bit stream for wl >= 7, the 32-bit stream below. */
int mv_block_quantize(const float* in, float* out, float* workspace, int64_t outer, int64_t dsize,
                      int64_t inner, int whole_tensor, int wl, int rounding, uint64_t seed,
                      uint64_t offset, void* stream);

/* debug: dump the 32-bit random stream the stochastic kernels consume for elements [0,n) */
int mv_philox_bits(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset, void* stream);
/* ... and the 16-bit stream of mv_float_quantize for man >= 7 (one value in [0, 65536) per element) */
int mv_philox_bits16(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset, void* stream);

/* weight_fake_quant for a Linear weight W fp32 [rows, cols] (torch.nn.qat.Linear.forward):
 * writes q(W) into `out` [rows, cols] and, if out_t != NULL, q(W)^T into out_t [cols, rows]
 * (the dgrad operand).  Container out_dtype: MV_F16 (exp<=5) or MV_F32. */
int mv_quantize_weight(const float* w, void* out, void* out_t, int out_dtype, int rows, int cols,
                       int exp_bits, int man_bits, void* stream);

/* ---------------------------------------------------------------- GEMM (tcgen05 / TMA)
 * C[M,N] = A * B^T over K, fp32 accumulate in TMEM, fused epilogue.
 *   a_major/b_major = 0: operand stored [M|N, K] row-major (K contiguous)   — forward, dgrad
 *                   = 1: operand stored [K, M|N] row-major (M|N contiguous) — wgrad (dY^T, X^T)
 *   a_dtype == b_dtype: MV_F16 (CTA-pair kernel, kind::f16) or MV_F32 (single-CTA kernel, kind::tf32);
 *   out_dtype: MV_F16 or MV_F32.  Any other type is an error.
 * Epilogue, in this order (each optional):
 *   acc (+ bias[n]) -> q_out -> [EPI_GELU: save u; acc = gelu(acc)] -> [EPI_DGELU: acc *= gelu'(u)]
 *   -> (+ residual[m,n]) -> q_res -> store out (out_dtype)
 *   accumulate != 0: out (fp32) += acc with red.global.add (split-K wgrad); bias/residual/q ignored.
 */
#define MV_EPI_NONE 0
#define MV_EPI_GELU 1   /* u = q_out(acc+bias); out = q_res(gelu(u)); aux (fp16 [M, ld_aux]) receives gelu'(u) */
#define MV_EPI_DGELU 2  /* acc *= aux[m,n]  (the gelu'(u) saved by the forward) */
/* rows_per_img > 0 (any epilogue): the residual is indexed by [m % rows_per_img, n] — the resized
 * positional embedding broadcast over the batch (models/vit.py:305-310). */

typedef struct {
    int M, N, K;
    const void* A; int lda; int a_dtype; int a_major;
    const void* B; int ldb; int b_dtype; int b_major;
    const float* bias;            /* [N] or NULL */
    const float* residual; int ld_res;   /* fp32 [M, ld_res] or NULL */
    void* aux; int ld_aux;        /* fp16, see MV_EPI_* */
    void* out; int ld_out; int out_dtype;
    int epilogue;
    int q_out_exp, q_out_man;     /* exp == 0: identity */
    int q_res_exp, q_res_man;
    int accumulate;               /* split-K atomic accumulation into fp32 `out` */
    int rows_per_img;             /* residual row = m % rows_per_img when > 0 */
    int tile_n;                   /* 0 = auto; 128 / 192 / 256 / 384 forces the tile width (testing; 384: split-K wgrad only) */
    float* colsum;                /* NULL, or fp32 [N]: colsum[n] += sum over m of the value stored to out[m, n] (fp32, before
                                   * the container rounding) with red.add — the bias gradient of the Linear whose output
                                   * gradient this GEMM produces, without a second pass over it.  CTA-pair kernel only. */
    int transpose_out;            /* accumulate only: out is [N, M] (pitch ld_out) and receives out[n, m] += acc[m, n].
                                   * CTA-pair kernel only. */
    /* Dropout (see "dropout mask" below); drop_seed == NULL: off.  The output [M, N] is the site tensor (C = N):
     * value (m, n) is multiplied by keep(seed, site, m*N + n) * drop_scale right after q_out — before the residual
     * add and q_res; in MV_EPI_GELU both gelu(u) and the stored gelu'(u) are multiplied before they are rounded, so the
     * MV_EPI_DGELU backward applies the mask without knowing about it.  CTA-pair kernel only, not with accumulate
     * or colsum. */
    const uint64_t* drop_seed;    /* device pointer to the 64-bit seed */
    uint32_t drop_thr;            /* keep when bits16 >= drop_thr; drop_thr = nearbyint(p * 65536) */
    float drop_scale;             /* 1 / (1 - p) in fp32 (0 for p == 1) */
    int drop_site;
    /* q_out rounded stochastically (see "gradient rounding stream" below); round_seed == NULL: nearest.  Value (m, n) of
     * the output [M, N] is element i = m*N + n of the site tensor, rounded to (q_out_exp, q_out_man), which must be a
     * float format, with the bits that mv_float_quantize(..., MV_ROUND_STOCHASTIC, *round_seed, round_offset) uses for
     * element i.  The rounding takes q_out's place in the epilogue (before the gelu' multiply of MV_EPI_DGELU).  An fp16
     * output raises the overflow flag where the value before or after rounding does not fit fp16.  CTA-pair kernel only,
     * plain or MV_EPI_DGELU outputs (colsum allowed; no accumulate, residual or dropout). */
    const uint64_t* round_seed;   /* device pointer to the 64-bit seed */
    uint64_t round_offset;
} mv_gemm_args;

int mv_gemm(const mv_gemm_args* args, void* stream);

/* ---------------------------------------------------------------- overflow sink
 * Replaces the inf / NaN test of torch.cuda.amp.GradScaler (classification/train.py:167, 259-277; the reference
 * trains under GradScaler(65536) and skips a step whose gradients are not finite).  flag_dev: one device int (or
 * NULL to switch reporting off, the default).  It is raised (set to 1, never cleared by the library) when
 *   - a value that a backward kernel rounds into an fp16 operand container does not fit it (|v| >= 65520: the
 *     container saturates at 65504): mv_scale_f32's fp16 copy, mv_layernorm_q_bwd's dx_f16, 16-bit outputs of
 *     mv_gemm that carry no quantiser (dgrad / gelu' outputs; the unquantised qkv of FP16_32), dqkv of
 *     mv_attention_bwd;
 *   - mv_scale_f32 meets a non-finite result (the un-scale pass over the parameter gradients sees every NaN / inf
 *     the backward produced; each element is tested, so a finite FLT_MAX does not raise it).
 * The caller clears it at the start of a step and hands it to mv_adamw_step's found_inf (no host sync).
 * The library does not own the int: it keeps the one pointer process-wide and every later launch of the kernels
 * above, by any caller, writes through it.  Register it only around the launches that should report into it, and
 * unregister it (NULL) before the int is freed.  A launch captured into a CUDA graph keeps the pointer it was
 * captured with. */
int mv_set_overflow_flag(int* flag_dev);
/* End-of-step bookkeeping, GradScaler.update() on the device: state_dev = {found_inf, scale_target, good_steps}
 * (3 floats).  found_inf <- found_inf (sticky until the caller clears it) or flag != 0 or *shared_slot != 0 (shared_slot, nullable: a float that went through the
 * gradient all-reduce, so that every rank of a data-parallel job sees every rank's flag); on found_inf
 * scale_target <- max(scale_target * backoff, min_target), else after growth_interval clean steps
 * scale_target <- min(scale_target * growth, max_target).  scale_target is the magnitude the backward scales the
 * largest incoming gradient to before it enters fp16 operand containers. */
int mv_overflow_update(const int* flag_dev, const float* shared_slot_dev, float* state_dev, float backoff, float growth,
                       int growth_interval, float min_target, float max_target, void* stream);


/* ---------------------------------------------------------------- LayerNorm + quant (warp-shuffle)
 * y = q_post(LN(q_in(x); gamma, beta)) : Sequential(QuantStub, nn.LayerNorm) followed by the next
 * Linear's QuantStub (models/vit.py:37-41; utils/quantize.py:215-220).  One warp per row.
 * y container: MV_F16 (formats that fit fp16) or MV_F32.  mean/rstd (fp32 [rows]) are saved for backward. */
int mv_layernorm_q_fwd(const float* x, int64_t ld_x, const float* gamma, const float* beta, void* y,
                       int64_t ld_y, int y_dtype, float* mean, float* rstd, int rows, int D, float eps,
                       int q_in_exp, int q_in_man, int q_post_exp, int q_post_man, void* stream);
/* dx = LN'(dy; q_in(x)) [-> q_grad] + dres (dres nullable); dx_f16 (nullable) gets an fp16 copy of dx (the next GEMM
 * operand).  dgamma/dbeta/dbias_prev (fp32 [D], nullable) are ACCUMULATED (+=): sum dy*xhat, sum dy, sum dx. */
typedef struct {
    const void* dy; int dy_dtype; int64_t ld_dy;   /* MV_F32 or MV_F16 (the dgrad GEMM's output) */
    const float* x; int64_t ld_x;
    const float* dres; int64_t ld_dres;
    const float* gamma; const float* mean; const float* rstd;
    float* dx; int64_t ld_dx;
    void* dx_f16; int64_t ld_lp;
    float* dgamma; float* dbeta; float* dbias_prev;
    int rows, D;
    int q_in_exp, q_in_man;
    /* Gradient quantiser (QPyTorch's Quantizer(backward_number=FloatingPoint(exp, man)), qtorch/quant/quant_module.py — an
     * option the reference's NumberFormat.quantizer never sets, utils/quantize.py:47-72): exp == 0: off; otherwise exp
     * 2..8, man 1..22.  It rounds the LayerNorm-input gradient (the backward of the QuantStub in front of the LayerNorm)
     * before dres is added; the stubs in front of the Linears are the q_out of their dgrad mv_gemm, the weight quantisers
     * a mv_float_quantize over the accumulated weight gradient (the caller passes them: mv_engine.EncoderEngine.backward). */
    int q_grad_exp, q_grad_man;
    /* round_seed (device pointer) != NULL: the gradient quantiser rounds stochastically with the "gradient rounding
     * stream" (element i = row*D + c; see below); NULL: nearest.  No effect without a gradient format. */
    const uint64_t* round_seed; uint64_t round_offset;
    /* Dropout (see "dropout mask"); drop_seed == NULL: off.  The mask (site drop_site) is applied to what feeds the Linear
     * in front of the residual stream: dx_f16 and the dbias_prev column sums get keep * drop_scale times dx; the fp32 dx
     * (the residual gradient) stays unmasked unless mask_dx != 0 (then every output is masked: the embedding site). */
    const uint64_t* drop_seed; uint32_t drop_thr; float drop_scale; int drop_site; int mask_dx;
} mv_layernorm_bwd_args;
/* The gradient quantiser and dropout take fp16 dy. */
int mv_layernorm_q_bwd(const mv_layernorm_bwd_args* args, void* stream);
/* out[c] += sum_r in[r,c]   (bias gradients); in_dtype MV_F16 or MV_F32 */
int mv_colsum(const void* in, int in_dtype, int64_t ld, int rows, int cols, float* out, void* stream);
/* img NCHW fp32 -> q(patches) [B*(H/P)*(W/P), P*P*C], (ph,pw,c) minor order (models/vit.py:271-275).
 * cls_slot = 1: each image gets one extra leading all-zero row (the class-token slot), so patch rows
 * line up 1:1 with token rows [B*N, .] for the embedding GEMM and its wgrad.  cls_slot = 2: a leading and a
 * trailing all-zero row per image (the class-token and distillation-token slots).  Any other value is an error. */
int mv_patchify_q(const float* img, void* out, int out_dtype, int B, int C, int H, int W, int P,
                  int q_exp, int q_man, int cls_slot, void* stream);
/* x[b,0,:] = q(q(cls) + pos_q[0,:]) for every image b (models/vit.py:283-310) */
int mv_cls_rows(const float* cls, const float* pos_q, float* x, int B, int n_tokens, int D, int q_exp,
                int q_man, void* stream);
/* x[b,row,:] = q(tok[:]) for every image b: the distillation token, which gets no positional embedding */
int mv_token_row(const float* tok, float* x, int B, int n_tokens, int D, int row, int q_exp, int q_man, void* stream);
/* out_f32[i] = in[i] * s and / or out_f16[i] = fp16_sat(in[i] * s) for n elements (n % 4 == 0; either output may
 * be NULL, out_f32 may alias in), s = *scale_dev or, with invert != 0, its reciprocal.  The backward's power-of-two
 * gradient scale is chosen on the device (no host sync); this applies / removes it in one pass. */
int mv_scale_f32(const float* in, const float* scale_dev, int invert, float* out_f32, void* out_f16, int64_t n,
                 void* stream);
/* ---------------------------------------------------------------- dropout mask
 * nn.Dropout(p) at a site of the encoder (the tensor is token-major [rows = B*N, cols = C]; element i = m*C + c):
 *   keep(seed, site, i) = bits16(seed, site, i) >= thr,   thr = (uint32) nearbyint(p * 65536)
 *   bits16 = half-word (i & 7) of Philox4x32-10(key = seed, counter = {i >> 3, site}) — the 16-bit stream of
 *            mv_float_quantize with offset = site (mv_philox_bits16 dumps it)
 *   D(y) = y * keep * scale,  scale = 1 / (1 - p) in fp32 (0 for p == 1); the drop probability is thr / 65536.
 * A pure function of (seed, site, m, c): forward, backward and the oracle see one mask whatever the tiling.
 * The seed is read from device memory (drawn per training forward from torch's generator), never a host constant.
 * Sites of encoder block l: 3l + 0 (to_out), 3l + 1 (after GELU), 3l + 2 (fc2); 3 * depth: after the positional add. */
/* out[rows, cols] = in * keep * scale; in / out MV_F32 or MV_F16 (each with its row pitch), in == out allowed.  An fp16
 * output saturates and raises the overflow flag (mv_set_overflow_flag) where |value| does not fit. */
int mv_dropout(const void* in, int in_dtype, int64_t ld_in, void* out, int out_dtype, int64_t ld_out, int rows, int cols,
               const uint64_t* seed_dev, int site, uint32_t thr, float scale, void* stream);
/* ---------------------------------------------------------------- gradient rounding stream
 * QPyTorch's Quantizer(backward_number=FloatingPoint(exp, man), backward_rounding="stochastic") at a gradient-quantiser
 * site: element i of the site tensor (token-major gradient [rows = B*N, cols = C]: i = m*C + c; a weight gradient: its
 * [out, in] layout) is rounded with the bits mv_float_quantize(x, exp, man, MV_ROUND_STOCHASTIC, seed, offset) uses for
 * element i — the 16-bit stream for man >= 7, the 32-bit stream for man < 7 — with
 *   offset = site + (rank << 32)   (rank: data-parallel rank, 0 on one GPU, so that ranks round independently)
 *   sites of encoder block l: 10l + k, k = 0 LN1 input, 1 to_qkv input, 2 to_qkv weight, 3 to_out input, 4 to_out
 *   weight, 5 LN2 input, 6 fc1 input, 7 fc1 weight, 8 fc2 input (before the gelu' multiply), 9 fc2 weight;
 *   10 * depth: the patch-embedding weight; 10 * depth + 1 + j: the decoder's quantisers in the order its forward
 *   applies them (the LayerNorm input first, then input and weight of each Linear).
 * The 64-bit seed is read from device memory (drawn per training forward from torch's generator, separate from the
 * dropout seed, whose sites use the same counter words).  The result is a pure function of (seed, offset, i): a fused
 * site equals mv_float_quantize_dev applied to the unfused value, bit for bit. */
/* mv_float_quantize with MV_ROUND_STOCHASTIC and the seed read from device memory (a captured CUDA graph rounds with
 * whatever seed the step drew). */
int mv_float_quantize_dev(const float* in, void* out, int out_dtype, int64_t n, int exp_bits, int man_bits,
                          const uint64_t* seed_dev, uint64_t offset, void* stream);
/* fp16 / fp32 in[rows, cols] (row pitch ld elements) times `mul` -> fp32 copy out[rows, cols] and / or
 * fp32 transpose out_t[cols, rows] with row pitch ld_t >= rows (either may be NULL).  The 32-bit formats (q_format TF32 / FP32) run
 * their contractions as kind::tf32 on K-major fp32 operands; this prepares dY^T / X^T for wgrad and
 * widens the fp16 attention tensors. */
int mv_widen_transpose(const void* in, int in_dtype, int64_t ld, int rows, int cols, float* out,
                       float* out_t, int64_t ld_t, float mul, void* stream);
/* 3xTF32 operand split for q_format FP32: in fp32 [rows, cols] (row pitch ld) -> out fp32 [rows, 3*cols] =
 * [hi | lo | hi] (mode 0, the A operand) or [hi | hi | lo] (mode 1, the B operand), hi = tf32 truncation of
 * x, lo = x - hi.  mv_gemm over the concatenated K computes hi*hi + lo*hi + hi*lo with fp32 accumulation
 * (product error ~2^-21), i.e. an fp32-grade Linear on the kind::tf32 tensor-core path. */
int mv_split_tf32(const float* in, int64_t ld, int rows, int cols, float* out, int mode, void* stream);

/* ---------------------------------------------------------------- attention (tcgen05, flash-style)
 * Attention.forward's (q @ k^T) * scale -> softmax -> @ v -> transpose/reshape (models/vit.py:87-97).
 * qkv: fp16 [B*N, 3*H*64] as written by the to_qkv GEMM (q | k | v, 64 columns per head).
 * out:  [B*N, H*64] container out_dtype, each value through q_out (the to_out QuantStub).
 * lse:  fp32 [B, H, N], log2-domain log-sum-exp of the scaled scores (saved for backward). */
int mv_attention_fwd(const void* qkv, void* out, int out_dtype, float* lse, int B, int H, int N,
                     float scale, int q_out_exp, int q_out_man, void* stream);
/* autograd backward of the above.  o: the saved forward output (fp16), d_o: fp16 gradient w.r.t. it,
 * delta: fp32 [B,H,N] scratch, dqkv: fp16 [B*N, 3*H*64] (dq | dk | dv).
 * dq_accum: fp32 [B*N, H*64] scratch: dQ is accumulated across key blocks with fp32 red.add.  Required when the
 * short-sequence kernel does not take the sequence (N > 272); an error if NULL there.
 * dbias: NULL or fp32 [3*H*64] (16-byte aligned): += the to_qkv Linear's bias gradient, i.e. the column sums of
 * dqkv.  The short-sequence kernel fuses it: the q part from the dQ rows it stores; the v part as the column sums
 * of d_o (sum_k dV[k,:] = sum_q (sum_k P[q,k]) dO[q,:] and the rows of P sum to one); the k part is left untouched
 * because it is identically zero (sum_k dS[q,k] = 0: a key bias shifts every score of a row alike).  Long
 * sequences take one mv_colsum pass over dqkv. */
int mv_attention_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, float* delta,
                     float* dq_accum, void* dqkv, float* dbias, int B, int H, int N, float scale, void* stream);

/* ---------------------------------------------------------------- optimizer step (SURVEY.md §8f.1)
 * Multi-tensor AdamW (torch.optim.AdamW / timm AdamW update rule, reference classification/train.py:
 * 161-166, 274-277) in ONE launch, fused with the weight fake-quantisation of the next step: for a
 * Linear weight (wq != NULL) the kernel also writes q(W) [rows, cols] and q(W)^T [cols, rows] in
 * the tensor-core operand container, replacing torch.nn.qat.Linear's per-forward weight_fake_quant.
 * `chunk0`: index of the tensor's first 1024-element chunk (a 32x32 tile for weights with wq); chunks
 * are numbered consecutively over the table and total_chunks is their sum.
 * hyper_dev (device, 6 floats): beta1, beta2, eps, step (>= 1), inv_scale (gradient un-scale),
 * found_inf (non-zero: parameters and moments untouched, operands still emitted). */
typedef struct {
    float* param;                 /* fp32 [n], updated in place */
    const float* grad;            /* fp32 [n] */
    float* exp_avg;               /* fp32 [n] */
    float* exp_avg_sq;            /* fp32 [n] */
    void* wq;                     /* NULL or q(W)   [rows, cols] */
    void* wq_t;                   /* NULL or q(W)^T [cols, rows] */
    int64_t n;
    int rows, cols;               /* rows * cols == n when wq != NULL */
    int wq_dtype;                 /* MV_F16 or MV_F32 */
    int q_exp, q_man;             /* weight format; q_exp == 0: identity */
    float lr, weight_decay;
    int chunk0;
} mv_adamw_tensor;
int mv_adamw_step(const mv_adamw_tensor* tensors_dev, int n_tensors, int total_chunks,
                  const float* hyper_dev, void* stream);

/* ---------------------------------------------------------------- low-precision optimizer (qtorch.optim.OptimLP)
 * mv_adamw_step with QPyTorch's OptimLP quantisers in the same single pass (DESIGN.md section 7).  For every element of
 * a tensor, unless found_inf is set:
 *   1. g = q_grad(grad * inv_scale * grad_scaling); grad_out (if not NULL) receives g
 *   2. the AdamW update of mv_adamw_step runs on acc (if not NULL) or on param itself, with gradient g
 *   3. exp_avg = q_exp_avg(exp_avg), exp_avg_sq = q_exp_avg_sq(exp_avg_sq)
 *   4. w = q_acc(updated value); acc (if not NULL) receives w
 *   5. param = q_weight(w); Linear weights (wq != NULL) emit q(W) / q(W)^T of this final param, as mv_adamw_step.
 * found_inf non-zero: nothing is written but the operands (grad_out included).
 * "Optimizer rounding stream": site s (0 grad, 1 exp_avg, 2 exp_avg_sq, 3 acc, 4 weight) of the tensor with `index` k
 * rounds element i (the tensor's flat row-major index, also for tiled Linear weights) stochastically with the bits that
 * mv_float_quantize(..., MV_ROUND_STOCHASTIC, seed, offset) (16-bit stream for man >= 7, else 32-bit stream) or
 * mv_fixed_point_quantize(..., MV_ROUND_STOCHASTIC, seed, offset) (32-bit stream) give element i, with
 *   offset = (step << 32) | (k << 3) | s,   step = hyper_dev[3] (1-based; a float, so exact below 2^24 steps).
 * The offset has no rank term: data-parallel ranks holding the same gradients round alike. */
#define MV_LPQ_NONE 0
#define MV_LPQ_FLOAT 1      /* FloatingPoint(exp_bits, man_bits): exp 1..8, man 1..22 (as mv_float_quantize) */
#define MV_LPQ_FIXED 2      /* FixedPoint(wl, fl, clamp, symmetric): wl 1..32, fl -100..100 (as mv_fixed_point_quantize) */
typedef struct {
    int kind;                     /* MV_LPQ_* */
    int rounding;                 /* MV_ROUND_NEAREST or MV_ROUND_STOCHASTIC */
    int exp_bits, man_bits;
    int wl, fl, clamp, symmetric;
} mv_lp_quant;
typedef struct {
    mv_lp_quant grad, exp_avg, exp_avg_sq, acc, weight;
    float grad_scaling;           /* multiplies the un-scaled gradient before q_grad */
    uint64_t seed;                /* Philox key of the optimizer rounding stream */
} mv_optim_lp;
/* per-tensor side table, one entry per mv_adamw_tensor (same order) */
typedef struct {
    float* acc;                   /* NULL: param is the accumulator; else fp32 [n], updated in place */
    float* grad_out;              /* NULL or fp32 [n] (may be grad itself): receives the quantised gradient */
    uint32_t index;               /* k: the parameter's position in the optimizer's flattened parameter list, < 2^29 */
} mv_adamw_lp_tensor;
int mv_adamw_lp_step(const mv_adamw_tensor* tensors_dev, const mv_adamw_lp_tensor* lp_dev, int n_tensors,
                     int total_chunks, const float* hyper_dev, const mv_optim_lp* spec, void* stream);

/* ---------------------------------------------------------------- segmentation loss (SURVEY.md §8f.4)
 * Fused nn.Upsample(size=(H, W), mode='bilinear', align_corners=False) + CrossEntropyLoss (reduction
 * 'mean', ignore_index) of the reference's segmentation head and train step (models/vit.py:355-371,
 * segmentation/train.py:188, 261), forward and backward in one pass; the [B, C, H, W] logits are never
 * materialised.  y, dy: fp32 [B, gh*gw, C] (patch-major, the decoder Linear's own output layout);
 * labels: int64 [B, H, W]; acc: fp32 [2], acc[0] += sum of pixel losses, acc[1] += non-ignored pixels;
 * dy += d(sum of pixel losses)/dy.  The caller zeroes dy / acc and divides by acc[1]. */
int mv_upsample_ce(const float* y, const int64_t* labels, float* dy, float* acc, int B, int C, int gh, int gw,
                   int H, int W, int64_t ignore_index, void* stream);

/* ---------------------------------------------------------------- distillation loss (DESIGN.md section 7)
 * The loss of DistillWrapper (models/distill.py), forward and backward in one pass over fp32 [B, C] student logits s,
 * distillation-head logits d and teacher logits t (row pitch C), int64 labels y [B]:
 *   row b:  ce = lse(s) - s[y],
 *           soft (hard == 0): D = T^2 * sum_c p_c (log p_c - log q_c),  p = softmax(t / T), q = softmax(d / T)
 *           hard (hard != 0): D = lse(d) - d[argmax t]  (the first maximal index, as torch.argmax)
 *   loss = (1 - alpha) * mean_b ce + alpha * mean_b D      (F.kl_div's "batchmean", F.cross_entropy's "mean")
 * d_student / d_distill (fp32 [B, C]) receive d loss / d s and d loss / d d; row_loss (fp32 [B]) is scratch that
 * receives each row's (1 - alpha) ce + alpha D.  The batch sum is a fixed-order reduction (no float atomics): the
 * result is deterministic.  A label outside [0, C) makes its row's loss and gradients NaN (no host sync to raise from;
 * the overflow sink of the backward then skips the step).  C >= 2, T > 0, 0 <= alpha <= 1.  Two launches. */
int mv_distill_loss(const float* student, const float* distill, const float* teacher, const int64_t* labels, int B,
                    int C, float T, float alpha, int hard, float* loss, float* row_loss, float* d_student,
                    float* d_distill, void* stream);

/* ---------------------------------------------------------------- Mixup / CutMix (DESIGN.md section 7)
 * timm 0.5.4's Mixup / mixup_target / SoftTargetCrossEntropy, with the randomness drawn on the device.  Image b is
 * mixed with its partner B - 1 - b (B even).  One "unit" is the whole batch (MV_MIX_BATCH), the pair {i, B - 1 - i}
 * (MV_MIX_PAIR, unit i < B / 2) or one image (MV_MIX_ELEM, unit b).  Per unit: with probability prob the unit is mixed
 * (else lam = 1, untouched); CutMix with probability switch_prob when both alphas are > 0, else the kind whose alpha is
 * > 0; lam ~ Beta(alpha, alpha) of that kind.
 *   Mixup:  pixel = fl32(fl32(w_self * a) + fl32(w_other * p)), w_self = fp32(lam), w_other = fp32(1 - lam) (fp64
 *           difference); a the image's pixel, p the partner's.
 *   CutMix: r = sqrt(1 - lam), cut_h = int(H r), cut_w = int(W r), cy ~ U{0..H-1}, cx ~ U{0..W-1},
 *           y0 = clip(cy - cut_h / 2, 0, H), y1 = clip(cy + cut_h / 2, 0, H) (x alike); pixels in [y0, y1) x [x0, x1)
 *           come from the partner and lam becomes 1 - (y1 - y0)(x1 - x0) / (H W).
 * "Mix stream": every draw of a unit is a Philox4x32-10 block with key = the 64-bit seed (device memory, drawn per
 * training forward from torch's generator) and counter = {unit, draw index, rank, MV_MIX_TAG}:
 *   draw 0:                  word 0: the mix test, 1: the CutMix switch, 2: cy, 3: cx (u = (word + 0.5) 2^-32)
 *   draw 1 + 17 g:           word 0: U of the alpha < 1 boost Gamma(alpha + 1) U^(1 / alpha) of Gamma draw g
 *   draw 2 + 17 g + k:       attempt k < 16 of Marsaglia-Tsang (fp64) for Gamma draw g: words 0, 1 a Box-Muller normal,
 *                            word 2 the acceptance test.  After 16 rejections the draw returns d = alpha' - 1/3
 *                            (times the boost); the probability of that is below 1e-20 for every alpha.
 *   lam = X / (X + Y) with X the Gamma draw g = 0, Y g = 1 (lam = 1/2 if both are 0).
 * rank (data-parallel rank) separates ranks that share the seed.  A pure function of (seed, rank, B, H, W, spec). */
#define MV_MIX_BATCH 0
#define MV_MIX_PAIR 1
#define MV_MIX_ELEM 2
#define MV_MIX_TAG 0x4d495855u
typedef struct {
    float mixup_alpha, cutmix_alpha;   /* >= 0, not both 0 */
    float prob, switch_prob;           /* in [0, 1] */
    int mode;                          /* MV_MIX_* */
} mv_mix_spec;
/* one per image */
typedef struct {
    float lam;                         /* target weight of the image's own label (after the CutMix correction) */
    float w_self, w_other;             /* the Mixup multipliers (1, 0 for CutMix and unmixed images) */
    int cutmix;                        /* 1: the box comes from the partner */
    int y0, y1, x0, x1;                /* the box (empty unless cutmix) */
} mv_mix_rec;
/* recs_dev: B records.  One launch. */
int mv_mix_draw(const int64_t* seed_dev, int rank, int B, int H, int W, mv_mix_spec spec, mv_mix_rec* recs_dev,
                void* stream);
/* mv_patchify_q of the mixed batch (the records applied to img before q_in), without materialising it.  A Mixup image
 * also reads its partner's rows, a CutMix image the partner's 16-byte vectors that overlap the box, an unmixed one
 * nothing more. */
int mv_patchify_mix_q(const float* img, const mv_mix_rec* recs_dev, void* out, int out_dtype, int B, int C, int H,
                      int W, int P, int q_exp, int q_man, int cls_slot, void* stream);
/* Soft-target cross-entropy over fp32 logits x [B, C] (row pitch C), int64 labels y [B]:
 *   t_b = lam_b s(y_b) + (1 - lam_b) s(y_{B-1-b}),  s(y) = off + (on - off) e_y,  off = smoothing / C,
 *   on = 1 - smoothing + off;   loss = mean_b sum_c -t_bc log_softmax(x_b)_c,   dlogits = (softmax(x) - t) / B.
 * recs_dev == NULL: lam = 1 (F.cross_entropy(x, y, label_smoothing=smoothing)).  row_loss: fp32 [B] scratch.  A label
 * outside [0, C) that carries weight (lam_b > 0 for y_b, lam_b < 1 for the partner's) makes the row's loss and
 * gradients NaN.  C >= 2, 0 <= smoothing <= 1, B even when recs_dev != NULL.  Fixed-order batch sum; two launches. */
int mv_mix_ce_loss(const float* logits, const int64_t* labels, const mv_mix_rec* recs_dev, int B, int C,
                   float smoothing, float* loss, float* row_loss, float* dlogits, void* stream);

/* ---------------------------------------------------------------- detection matching (SURVEY.md §8f.4)
 * scipy.optimize.linear_sum_assignment of the reference's HungarianMatcher (models/matcher.py:83-86) for a
 * whole batch in one launch, one warp per image.  cost: fp32 [B, Q, Tmax], image b uses columns
 * [0, sizes[b]); match: int32 [B, Tmax], match[b, t] = prediction matched to target t, -1 for padding
 * columns and for targets left over when sizes[b] > Q.  flag (may be NULL): set to 1 if some block has
 * no finite matching (SciPy raises there).  Q, Tmax <= 1024. */
int mv_linear_sum_assignment(const float* cost, const int* sizes, int B, int Q, int Tmax, int* match,
                             int* flag, void* stream);

/* ---------------------------------------------------------------- debug timelines
 * Only active in a library built with -DMV_SN_TRACE / -DMV_GEMM_TRACE (MV_NVCC_FLAGS for csrc/build.py):
 * CTA 0 of the short-sequence attention kernels / the CTA-pair GEMM writes {event, index, clock64} records
 * into dev_buf (int64 [3][1024][3]) at the hand-offs between its MMA issuer and its math / epilogue warps
 * (tools/trace_attn_bwd.py, tools/trace_gemm.py).  NULL switches recording off; no effect otherwise. */
int mv_debug_set_attn_trace(void* dev_buf);
int mv_debug_set_gemm_trace(void* dev_buf);

#ifdef __cplusplus
}
#endif
#endif /* MV_B200_H */
