/*
 * vl2.h — C-ABI of libvl2.so, the B200 (sm_100a) kernel library behind the VideoLLaMA2 video->text prefill path.
 *
 * The reference (DAMO-NLP-SG/VideoLLaMA2) is pure Python on top of HF transformers / timm / torch; it has no FFI.
 * Each entry point below therefore replaces a *library call site* of the reference hot path; the citation after
 * each declaration is the reference line (relative to /root/reference, or HF: = transformers/models) whose
 * arithmetic the call performs.  INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *  - extern "C", plain pointers + sizes; no torch types.  All data pointers are DEVICE pointers unless named host_*.
 *  - bf16 storage (`uint16_t`-sized), fp32 accumulate.  Row-major, leading dimensions in ELEMENTS.  The one exception is
 *    vl2_gemv_fp8, whose weights are fp8 E4M3 with a per-row fp32 scale (decode only; prefill weights stay 16-bit).
 *  - `stream` is a cudaStream_t passed as void*.  Calls enqueue work and return; they never synchronise, never
 *    allocate device memory, and are CUDA-graph capturable.
 *  - Every call returns 0 on success or a negative VL2_E_* code; vl2_last_error() gives a thread-local message.
 *  - There is no CPU fallback: on a machine without an sm_100 device the calls fail with VL2_E_CUDA.
 */
#ifndef VL2_H_
#define VL2_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VL2_VERSION 100

enum {
  VL2_OK = 0,
  VL2_E_BADSHAPE = -1,
  VL2_E_BADDTYPE = -2,
  VL2_E_BADALIGN = -3,
  VL2_E_CUDA = -4,
  VL2_E_NCCL = -5,
  VL2_E_UNSUPPORTED = -6
};

/* GEMM epilogue activations. */
enum {
  VL2_ACT_NONE = 0,
  VL2_ACT_QUICK_GELU = 1, /* x*sigmoid(1.702x)          HF:clip/modeling_clip.py:339-351 (quick_gelu)      */
  VL2_ACT_SILU = 2,       /* x*sigmoid(x)               projector.py:173 (nn.SiLU), timm LayerNormAct2d     */
  VL2_ACT_GELU_ERF = 3,   /* 0.5x(1+erf(x/sqrt2))       projector.py:128 (nn.GELU)                          */
  VL2_ACT_SWIGLU = 4,     /* out[:,j] = silu(acc[:,2j])*acc[:,2j+1]  HF:mistral/modeling_mistral.py:46-48   */
  VL2_ACT_GELU_TANH = 5   /* 0.5x(1+tanh(sqrt(2/pi)(x+0.044715x^3)))  HF SiglipMLP ("gelu_pytorch_tanh"), encoder.py:84-101 */
};

int vl2_version(void);
/* 16-bit storage type this build of the library moves through every `bf16` pointer of this header: 0 = bfloat16
 * (libvl2.so), 1 = IEEE float16 (libvl2_f16.so, the same sources compiled with -DVL2_HALF: the reference's own inference
 * dtype, videollama2/__init__.py:60).  Same entry points, same structs; accumulation is fp32 in both. */
int vl2_storage_dtype(void);
const char* vl2_last_error(void);
/* Number of kernel launches issued by this library in this process (bench.py's gpu_launches counter). */
int64_t vl2_launch_count(void);
/* Programmatic dependent launch for every subsequent vl2_* launch of this process: 1 = on (each kernel is launched with
 * the programmatic-stream-serialization attribute; kernels begin with griddepcontrol.launch_dependents and wait with
 * griddepcontrol.wait before touching their inputs, so a kernel's prologue - for the GEMV: the first weight-stage
 * prefetches - overlaps the tail of its predecessor), 0 = off, -1 = follow the VL2_PDL environment variable (default off).
 * Used by the single-token decode graph, where ~230 small kernels run back to back. */
int vl2_set_pdl(int mode);

/* ------------------------------------------------------------------------------------------------------------
 * Dense bf16 GEMM on tcgen05 tensor cores:  C[M,Nout] = epi( A[M,K] * W[N,K]^T ).
 *   epi(acc) = act( acc * row_scale[m] + bias[n] ) + residual[m,n]        (each term optional)
 *   VL2_ACT_SWIGLU: W rows interleave gate/up (row 2j = gate_j, row 2j+1 = up_j); Nout = N/2; residual unsupported.
 * Replaces nn.Linear / 1x1 nn.Conv2d / (after im2col) nn.Conv2d and nn.Conv3d call sites:
 *   HF:clip/modeling_clip.py:294-311,339-351 ; projector.py:153-187 (timm RegStage 1x1 convs, Conv3d, readout MLP) ;
 *   HF:mistral/modeling_mistral.py:35-48,122-177,402-470.
 * Requirements: K % 8 == 0, N % 8 == 0, lda/ldw/ldc/ldr % 8 == 0, pointers 16-byte aligned.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct vl2_gemm_args {
  const void* A;   /* bf16 [M,K]  */
  const void* W;   /* bf16 [N,K]  */
  void* C;         /* bf16 [M,Nout] (or fp32 if out_f32) */
  const float* bias;      /* fp32 [N] or NULL  */
  const void* residual;   /* bf16 [M,Nout] or NULL */
  const float* row_scale; /* fp32 [M] or NULL */
  int64_t lda, ldw, ldc, ldr;
  int32_t M, N, K;
  int32_t act;
  int32_t out_f32;
  int32_t reserved; /* 0 = choose the tile by the library's cost model; 64..256 (step 32) forces a single-CTA tile width,
                       1000 + (128..256) forces the cta_group::2 pair kernel (tests) */
  /* Fused compute + collective (frame-parallel ViT, SURVEY.md §8e): every output vector of C is ALSO stored at the same
   * element offset into up to 8 peer buffers (other GPUs' symmetric memory mapped over NVLink), or once to an NVSwitch
   * multicast address (multimem.st) when mc_out != NULL — the all-gather of visual tokens happens inside the epilogue
   * of the producing GEMM, tile by tile, instead of in a separate collective.  bf16, non-SwiGLU outputs only. */
  void* bcast_out[8];
  void* mc_out;
  int32_t n_bcast;
  int32_t reserved2;
  /* RMSNorm folded into the GEMMs around it (HF:mistral/modeling_mistral.py:182-199): with gamma pre-multiplied into
   * W's columns, rmsnorm(x) W^T = rsqrt(mean(x^2) + eps) * (x W'^T).
   *   rms_sumsq_in  fp32 [M, rms_nparts]: partial sums of squares of THIS GEMM's A rows (summed in a fixed order) ->
   *                 the accumulator is scaled by rsqrt(sum_p rms_sumsq_in[m,p] * rms_inv_dim + rms_eps) before
   *                 bias/activation (NULL = off)
   *   sumsq_out     fp32 [M, N/32]: the epilogue writes, per 32 output columns, sum C[m,n]^2 of the bf16-rounded outputs
   *                 (a 64-column span writes its sum to the first slot and 0 to the second): the next norm's statistics
   *                 come for free from the producing residual GEMM, with no atomics (bit-reproducible). */
  const float* rms_sumsq_in;
  float* sumsq_out;
  int32_t rms_nparts;
  int32_t reserved3;       /* test hook: 2..4 forces that many K-slices for the tiles of the last round (needs splitk_ws) */
  float rms_inv_dim;
  float rms_eps;
  /* optional split-K workspace (device memory, 16-byte aligned, ZERO-FILLED once by the caller, reusable by every later
   * launch on the same stream): when the tile count leaves the last round of the persistent grid mostly idle, the
   * remaining tiles are cut into K-slices whose fp32 partial accumulators go through this buffer (deterministic order).
   * 64 KB of counters + up to ~40 MB of partials; NULL / too small = no split.  Opt-in (environment VL2_GEMM_SPLITK=1): on
   * the 7B shapes it pays only for K = 14336 and it makes rounding depend on M; see DESIGN.md. */
  void* splitk_ws;
  int64_t splitk_ws_bytes;
  /* LayerNorm folded into the GEMMs around it (HF:clip/modeling_clip.py:354-385 layer_norm1 / layer_norm2 in front of
   * q/k/v_proj and fc1): with W' = W * gamma (columns), colsum[n] = sum_k W'[n,k] and bias' = bias + W beta,
   *     LN(x; gamma, beta) W^T + bias = rstd * (x W'^T - mu * colsum) + bias'.
   *   ln_sum_in     fp32 [M, rms_nparts]: partial row sums of THIS GEMM's A rows; together with rms_sumsq_in (the partial
   *                 sums of squares, REQUIRED with it) they give mu = sum/K and rstd = rsqrt(max(E[x^2] - mu^2, 0) + rms_eps);
   *                 the accumulator becomes (acc - mu * ln_colsum[n]) * rstd before bias/activation (NULL = off)
   *   ln_colsum     fp32 [N] (REQUIRED with ln_sum_in)
   *   rowsum_out    fp32 [M, N/32]: like sumsq_out, the per-32-column sums of the bf16-rounded outputs (NULL = off; same
   *                 restrictions as sumsq_out) */
  const float* ln_sum_in;
  const float* ln_colsum;
  float* rowsum_out;
  /* Implicit-GEMM front end for nn.Conv3d(C, N, kernel_size = stride = 2, padding = conv_pad) on channels-last input
   * (projector.py:164-174, the STC connector's sampler; SURVEY.md Appendix A): with conv_C > 0, A is NOT a matrix but the
   * activation x bf16 [conv_T, conv_H, conv_W, conv_C]; W is the kernel as [N, 8*conv_C] with K index = tap*C + cin,
   * tap = dt*4 + dh*2 + dw; M must equal To*Ho*Wo and K = 8*conv_C; C rows are the output positions (to, ho, wo) row-major.
   * The TMA producer gathers each k-block (one tap x 64 channels) of 8 output lines straight from x with ONE box of a 5-D
   * tensor map over x viewed as [T, H/2, 2, W/2, 2C] (out-of-bounds = the zero padding): no im2col matrix exists.
   * Up to 16 x 16 output positions per time step; odd H / W only with conv_pad = 0.  lda is ignored.  bias + activation
   * epilogues only.  reserved4: 0; test hook 1 = use the general epilogue where the lean (TMA-store) one would be
   * picked (both are parity-tested against each other). */
  int32_t conv_C, conv_T, conv_H, conv_W, conv_pad, reserved4;
  /* RoPE in the epilogue of the fused QKV projection (HF:mistral/modeling_mistral.py:51-82 apply_rotary_pos_emb): output
   * columns [0, rope_cols) are q and k heads of width rope_D whose weight rows were permuted at load so that the rotation
   * partners (i, i + D/2) of a head are ADJACENT output columns (2i, 2i+1); the epilogue rotates each pair of row m with
   * the angle of position rope_pos0 + m and frequency i:  (a, b) -> (a cos - b sin, b cos + a sin).  q.k dot products are
   * invariant under the (consistent) permutation, so attention and the KV cache need no un-permute.
   *   rope_tab  uint32 [positions, rope_D/2]: bf16 cos in the low half, bf16 sin in the high half (HF rounds cos/sin to
   *             the activation dtype), device memory; NULL = off.  bf16 output, no activation. */
  const uint32_t* rope_tab;
  int32_t rope_cols, rope_D, rope_pos0, reserved5;
} vl2_gemm_args;
int vl2_gemm_bf16(const vl2_gemm_args* args, void* stream);
/* Debug aid: with args->reserved2 == 777 CTA 0 records clock64() at its tile boundaries: out[0] = tiles traced (<= 7), and
 * for tile t at out[8t+1..8t+6]: MMA role waits for the accumulator stage / starts issuing / issued its last commit;
 * epilogue warp starts the tile / sees the accumulator complete / stored its last span; out[64+8t .. 64+8t+5]: phases of that
 * warp's first 64-column span (start, residual staged, accumulator chunk loaded, first / second half computed, stored).
 * host_out128: 128 values.  Synchronises the device. */
int vl2_debug_gemm_trace(long long* host_out128);
/* Planning only, no device work: out6 = {tile width BN, 1 if the 256-row cta_group::2 tile is used, number of tiles,
 * CTAs (or CTA pairs) the persistent grid runs, rounds = ceil(tiles / that), SM count assumed (148 without a device)}. */
int vl2_gemm_plan(int M, int N, int K, int with_splitk_ws, int32_t* out6);

/* Skinny GEMM (M <= 32 rows, HBM-bound weight streaming): C[M,N] = act(A[M,K] W[N,K]^T + bias).
 * Used for the SE excitation MLP of the RegStage blocks (timm SEModule, projector.py:153-161) and the last-position
 * lm_head GEMV (HF:mistral/modeling_mistral.py:463-466 with logits_to_keep=1).  act_out: VL2_ACT_NONE/SILU or
 * 100 = sigmoid, or VL2_ACT_SWIGLU (interleaved gate/up rows -> N/2 outputs).  C is fp32 if out_f32 else bf16; A is fp32
 * if a_f32 else bf16.  With M = 1 this is every linear layer of a KV-cache decode step (HBM-bound weight streaming). */
int vl2_gemm_skinny(const void* A, int a_f32, const void* W, const float* bias, const void* residual /* bf16 [M,N] or NULL */,
                    void* C, int out_f32, int M, int N, int K, int act, void* stream);

/* GEMV, the M = 1 case of the above as its own entry point (every nn.Linear of a single-token decode step):
 * y[N] = act(s * W[N,K] x + bias) (+ residual); with rms_eps > 0, s = rsqrt(mean(x^2) + rms_eps): the RMSNorm in front of
 * the projection (HF:mistral/modeling_mistral.py:35-48) with its gain folded into W's columns, at no extra pass over x.
 * act as vl2_gemm_skinny.  HBM-bound: 2*N*K bytes. */
int vl2_gemv_bf16(const void* x, const void* W, const float* bias, const void* residual /* bf16 [N] or NULL */, void* y,
                  int out_f32, int N, int K, int act, float rms_eps, void* stream);
/* The same GEMV with fp8 weights (opt-in decode weights, `decode_weights="fp8"`): W8 is fp8 E4M3 [N,K] (no NaN codes) and
 * w_scale fp32 [N] its per-row dequantisation scale, y[N] = act(w_scale[n] * s * W8[n,:] x + bias) (+ residual); with
 * VL2_ACT_SWIGLU the gate and up rows each carry their own scale.  x, residual and y are the build's 16-bit type.
 * Requirements: K % 16 == 0, w_scale != NULL, x / W8 16-byte aligned.  HBM-bound: N*K bytes, half of vl2_gemv_bf16's. */
int vl2_gemv_fp8(const void* x, const void* W8, const float* w_scale, const float* bias,
                 const void* residual /* bf16 [N] or NULL */, void* y, int out_f32, int N, int K, int act, float rms_eps,
                 void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Fused attention (FlashAttention-style, tcgen05 QK^T / PV with TMEM accumulators, TMA-staged K/V).
 *   q: bf16 [B*S, ldq] with head h at columns [q_off + h*D, +D)   (likewise k, v with kv head h / (Hq/Hkv))
 *   out: bf16 [B*S, ldo], head h at columns [h*D, +D).  softmax scale applied to logits in fp32.
 * causal = 0: HF:clip/modeling_clip.py:282-336 (CLIPAttention, 16 heads x 64).
 * causal = 1: HF:mistral/modeling_mistral.py:122-177 / qwen2/modeling_qwen2.py:187-246 (GQA, D=128).
 * D: any multiple of 8 up to 128 (64 / 128 natively; other widths, e.g. SigLIP-so400m 72, run the next wider kernel with
 * TMA zero fill beyond the head, heads packed at their true width in memory).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct vl2_attn_args {
  const void* q;
  const void* k;
  const void* v;
  void* out;
  int64_t ldq, ldk, ldv, ldo; /* row strides in elements */
  int32_t B, S, Hq, Hkv, D;
  int32_t causal;
  float scale;
  int32_t reserved;
} vl2_attn_args;
int vl2_attention(const vl2_attn_args* args, void* stream);
/* Debug aid: with args->reserved == 777 one softmax thread of CTA (0,0,0) accumulates the cycles it spends in each
 * phase of the key-tile loop; this call synchronises the device and copies the 16 counters to host memory
 * ([0] wait S, [1] TMEM load, [2] mask+max+exchange, [3] wait PV / rescale, [4] exp2+pack+st.shared, [5] fence+arrive,
 *  [6] item epilogue, [7] key tiles traced, [8] work items traced, [9] cycles of the CTA's whole item loop);
 * reserved == 778 traces every work item of the persistent CTA 0 instead of its first (cold) one. */
int vl2_debug_attn_trace(long long* host_out16);
/* Debug aid: with args->reserved == 779 the softmax thread, the MMA-issuing thread and the two TMA producer lanes of the
 * persistent CTA 0 stamp clock64() at every hand-over of its second work item (slot map: csrc/attn_tcgen05.cu,
 * g_attn_tl); this call synchronises the device and copies the 320 stamps to host memory (tools/attn_trace.py). */
int vl2_debug_attn_timeline(long long* host_out320);

/* Hint: pull [ptr, ptr + bytes) into L2 (cp.async.bulk.prefetch.L2 in 16 KB pieces; returns immediately).  The decode graph
 * forks this next to the latency-bound attention phase so the o_proj / gate-up GEMVs start from L2-resident weights. */
int vl2_l2_prefetch(const void* ptr, size_t bytes, void* stream);

/* Single-token decode attention over a KV cache (HF:mistral/modeling_mistral.py:122-177 with a DynamicCache):
 * q bf16 [Hq*D]; k_cache / v_cache bf16 rows of ldkv elements (kv head h at columns [h*D, +D)), positions 0..n_pos-1;
 * out bf16 [Hq*D].  Split over the KV length (flash-decoding): `workspace` is a caller-owned device buffer of
 * vl2_attention_decode_workspace(Hq, Hkv, D) bytes holding the per-split partial results.  Hq/Hkv <= 8. */
size_t vl2_attention_decode_workspace(int Hq, int Hkv, int D);
int vl2_attention_decode(const void* q, const void* k_cache, const void* v_cache, void* out, int64_t ldkv, int n_pos,
                         int Hq, int Hkv, int D, float scale, void* workspace, void* stream);
/* CUDA-graph-replayable decode step: the current position is read from DEVICE memory (*pos_dev), so one captured graph
 * serves every token.  vl2_decode_rope_append rotates q/k of the freshly projected fused row [q|k|v] at position *pos_dev
 * and copies the row into cache[*pos_dev]; vl2_attention_decode_dyn attends to cache rows 0..*pos_dev and is
 * bit-identical to vl2_attention_decode(n_pos = *pos_dev + 1). */
int vl2_decode_rope_append(void* qkv_row, void* cache, int64_t cache_ld, const int32_t* pos_dev, int Hq, int Hkv, int D,
                           const float* inv_freq, int interleaved /* pairing, see vl2_rope_inplace */, void* stream);
int vl2_attention_decode_dyn(const void* q, const void* k_cache, const void* v_cache, void* out, int64_t ldkv,
                             const int32_t* pos_dev, int Hq, int Hkv, int D, float scale, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Row-wise normalisations (HBM-bound, one pass).
 * vl2_layernorm: y = act( LN(x; gamma, beta, eps) [+ residual] )  over the last dim C (bf16 in/out, fp32 math).
 *   act in {NONE, SILU}; with residual the order is act(LN(x) + residual)   (timm Bottleneck: act3(conv3(..)+shortcut)).
 *   HF:clip/modeling_clip.py:363-385 (layer_norm1/2, pre_layrnorm) ; timm LayerNormAct2d inside RegStage.
 * vl2_rmsnorm:   y = bf16( x * rsqrt(mean(x^2)+eps) ) * gamma     HF:mistral/modeling_mistral.py:182-199.
 * ---------------------------------------------------------------------------------------------------------- */
int vl2_layernorm(const void* x, const void* gamma, const void* beta, const void* residual, void* y, int64_t rows,
                  int C, float eps, int act, void* stream);
int vl2_rmsnorm(const void* x, const void* gamma, void* y, int64_t rows, int C, float eps, void* stream);
/* out[r] = sum_c x[r,c]^2 (fp32): seeds the folded-RMSNorm statistics for the first decoder layer. */
int vl2_row_sumsq(const void* x, float* out, int64_t rows, int C, void* stream);
/* Row sums AND row sums of squares (fp32 [rows] each): the statistics of a LayerNorm folded into the consuming GEMM
 * (vl2_gemm_args.ln_sum_in / rms_sumsq_in) when the rows were not produced by a GEMM epilogue, e.g. the output of
 * pre_layrnorm in front of CLIP's first encoder layer (HF:clip/modeling_clip.py:354-385). */
int vl2_row_stats(const void* x, float* sum_out, float* sumsq_out, int64_t rows, int C, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * CLIP patch embedding front/back ends (HF:clip/modeling_clip.py:202-218).
 * vl2_patch_im2col: pixels bf16 [F,3,H,W] (NCHW) -> A bf16 [F*(H/P)*(W/P), Kpad], column = c*P*P + i*P + j, zero
 *   padded to Kpad (Kpad % 64 == 0) so the patch conv becomes vl2_gemm_bf16 against weight[1024, Kpad].  H / P and
 *   W / P round down like the strided conv does (SigLIP@384, P = 14: 27 x 27 patches, the last 6 pixels are unused).
 * vl2_clip_embed_finish: tok[f, 0] = cls + pos[0]; tok[f, 1+p] = patch[f*np+p] + pos[1+p]; then pre_layrnorm.
 * ---------------------------------------------------------------------------------------------------------- */
int vl2_patch_im2col(const void* pixels, void* A, int F, int H, int W, int P, int Kpad, void* stream);
int vl2_clip_embed_finish(const void* patch, const void* cls, const void* pos, const void* gamma, const void* beta,
                          void* tok, int F, int np, int C, float eps, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * STC connector pieces (projector.py:133-215; timm regnet.Bottleneck), channels-last [F,H,W,C].
 * vl2_dwconv3x3_ln_silu: y = SiLU(LN_c(depthwise3x3(x; w[9,C]))); if pooled != NULL it must hold F*C + F*H*C floats:
 *   pooled[0 : F*C] receives mean_{h,w} y[f,h,w,c] (the SE squeeze), the rest is workspace for per-row partial sums
 *   (deterministic two-step reduction, no atomics).
 * vl2_se_scale: y[f,p,c] *= s[f,c]  (s fp32 [F,C]).
 * vl2_conv3d_im2col: A[(t',h',w'), tap*C + c] = x[2t'-1+dt+pad.., ...] for the k=s=2 Conv3d with padding `pad`
 *   (1 for stc_connector, 0 for stc_connector_v35); OOB taps are zero.  Then vl2_gemm_bf16 with W[C, 8C].
 * ---------------------------------------------------------------------------------------------------------- */
int vl2_dwconv3x3_ln_silu(const void* x, const void* w9c, const void* gamma, const void* beta, void* y, float* pooled,
                          int F, int H, int W, int C, float eps, void* stream);
int vl2_se_scale(void* y, const float* s, int F, int HW, int C, void* stream);
int vl2_conv3d_im2col(const void* x, void* A, int T, int H, int W, int C, int pad, int To, int Ho, int Wo,
                      void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Decoder glue.
 * vl2_rope_inplace: rotate-half RoPE on q and k heads inside a fused [S, ld] QKV buffer, positions pos0..pos0+S-1.
 *   HF:mistral/modeling_mistral.py:51-82,262-323 (cos/sin in fp32 from inv_freq = theta^(-2i/D)).
 * vl2_embed_splice: inputs_embeds[dst_row[i]] = table[ids[i]] for text positions (ids >= 0); visual rows are written
 *   directly by the readout GEMM.  videollama2_arch.py:198-220.
 * ---------------------------------------------------------------------------------------------------------- */
int vl2_rope_inplace(void* qkv, int64_t ld, int S, int Hq, int Hkv, int D, int q_off, int k_off, int pos0,
                     const float* inv_freq /* fp32 [D/2], device */,
                     int interleaved /* 0: HF rotate-half pairing (i, i + D/2); 1: pairs are adjacent columns (2i, 2i+1) -
                                        the layout of a QKV projection whose q/k weight rows were permuted for the
                                        RoPE-in-epilogue GEMM (vl2_gemm_args.rope_tab) */,
                     void* stream);
int vl2_embed_splice(const int64_t* ids, const int32_t* dst_row, int n, const void* table, int64_t vocab, void* out,
                     int H, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Frame preprocessing on the device (the step in front of the tower: videollama2/mm_utils.py:27-38 expand2square,
 * :91-103 process_image, :132-202 process_video -> transformers 4.40 CLIPImageProcessor / SiglipImageProcessor ->
 * Pillow Image.resize(BICUBIC)).  uint8 RGB frames [T,H,W,3] are placed (virtually) on a canvas_h x canvas_w canvas filled
 * with pad_rgb at offset (off_y, off_x), resized to out_h x out_w with Pillow's two-pass fixed-point antialiased bicubic
 * resampler (bit-exact: the 22-bit coefficient tables bounds_* [n,2] = (first tap, taps), kk_* [n, ksize_*] are computed by
 * the caller exactly as Resample.c does), cropped to crop x crop at (crop_top, crop_left), mapped through lut [3,256]
 * (= (u8 * (1/255) - mean) / std in float32) and stored as bf16 [T,3,crop,crop]; out_u8 (optional) receives the resized
 * uint8 window [T,crop,crop,3].  tmp: vl2_preprocess_workspace() bytes.  HBM-bound byte work.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct vl2_preprocess_args {
  const uint8_t* frames;
  int32_t T, H, W;
  int32_t canvas_h, canvas_w, off_y, off_x;
  uint8_t pad_rgb[4];
  int32_t out_h, out_w;
  int32_t crop_top, crop_left, crop;
  const int32_t* bounds_h;
  const int32_t* kk_h;
  const int32_t* bounds_v;
  const int32_t* kk_v;
  int32_t ksize_h, ksize_v;
  const float* lut;
  uint8_t* tmp;
  void* out_bf16;
  uint8_t* out_u8;
} vl2_preprocess_args;
size_t vl2_preprocess_workspace(const vl2_preprocess_args* args);
int vl2_preprocess_frames(const vl2_preprocess_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * ViT patch embedding as one implicit-GEMM kernel (HF CLIPVisionEmbeddings.forward + pre_layrnorm,
 * HF:clip/modeling_clip.py:202-218,739-741; HF SiglipVisionEmbeddings for encoder.py:84-151):
 *   CLIP   (gamma != NULL): out[f, 0] = LN(cls + pos[0]);  out[f, 1+p] = LN(conv(pixels[f])[p] + pos[1+p])
 *   SigLIP (gamma == NULL): out[f, p] = conv(pixels[f])[p] + bias + pos[p]
 * pixels bf16 [F,3,H,W]; weight bf16 [C, Kpad] = patch_embedding.weight flattened (c, i, j)-major and zero-padded from
 * 3*P*P to Kpad (multiple of 64, <= 640); pos bf16 [np (+1), C]; out bf16 [F*(np (+1)), C].  The A operand is gathered
 * from the frames by the kernel (LDG -> 128B-swizzled shared memory); no im2col matrix exists.  A 128-patch row block is
 * split along C over a thread-block cluster of up to 4 CTAs that keep their accumulators in TMEM and exchange the
 * LayerNorm statistics through distributed shared memory: nothing un-normalised leaves the SM (`scratch` is unused).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct vl2_patch_embed_args {
  const void* pixels;
  const void* weight;
  const void* pos;
  const void* cls;     /* bf16 [C] (CLIP) or NULL */
  const void* gamma;   /* pre_layrnorm weight / bias (CLIP) or NULL */
  const void* beta;
  const float* bias;   /* conv bias fp32 [C] (SigLIP) or NULL */
  void* out;
  float* scratch;      /* unused (kept for ABI stability) */
  int32_t F, H, W, P, C, Kpad;
  float eps;
  int32_t reserved;
} vl2_patch_embed_args;
int vl2_patch_embed(const vl2_patch_embed_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Tensor-parallel decoder (BASELINE.json configs[4], SURVEY.md §8e "TP decoder"; no counterpart in the reference, whose
 * multi-GPU loading is accelerate's device_map="auto", videollama2/model/__init__.py:48,54):
 * all-reduce of the row-parallel GEMMs' bf16 partials [S,H] over the ranks of one NVSwitch domain, fused with the row sums
 * of squares the next folded RMSNorm needs, as ONE kernel with its cross-GPU barriers inside.  All buffers are symmetric
 * memory (the same allocation on every rank, peer-mapped over NVLink): part[r] / xout[r] / stats[r] / pads[r] are rank r's
 * buffers as seen from THIS rank; *_mc are the NVSwitch multicast addresses of the same buffers (NULL = no multicast: the
 * kernel broadcasts with peer stores instead of multimem.st).  Rank r reduces rows
 * [r*ceil(S/world), ...) and writes them to every rank.  pads: >= 17 zero-initialised uint32 per rank; `epoch` = 1, 2, 3, ...
 * counts the calls that used these pads (the same on every rank).  Not CUDA-graph replayable (epoch is a launch argument).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct vl2_tp_allreduce_args {
  const void* part[8];
  void* xout[8];
  float* stats[8];
  uint32_t* pads[8];
  const void* part_mc;
  void* xout_mc;
  float* stats_mc;
  int32_t rank, world, S, H;
  uint32_t epoch;
  uint32_t inswitch_reduce; /* 1: reduce inside the NVSwitch (multimem.ld_reduce; needs *_mc).  Off by default: measured on
                               B200 the switch does not round bf16 sums to nearest (1-ulp differences on ~19 % of the
                               elements), so the default reduces with peer loads (exact fp32 accumulation) and uses the
                               switch for the broadcast only */
} vl2_tp_allreduce_args;
int vl2_tp_allreduce_stats(const vl2_tp_allreduce_args* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VL2_H_ */
