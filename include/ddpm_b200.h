/* ddpm_b200 — C ABI of the B200-native DDPM engine (libddpm_b200.so).
 *
 * The reference (tqch/ddpm-torch @ b60eb8d) is pure Python on PyTorch and has NO FFI / plugin interface;
 * its seam for this path is the Python callable protocol  denoise_fn(x_t f32[B,C,H,W], t i64[B]) -> f32[B,C,H,W]
 * (ddpm_torch/diffusion.py:109,238; ddim.py:101) plus the GaussianDiffusion / DDIM methods that call it.
 * This header is what a ctypes binding on the reference side binds instead (see INTEGRATION.md); every entry
 * point cites the reference code it replaces.
 *
 * Conventions
 *  - plain pointers and sizes only; all pointers are DEVICE pointers unless stated otherwise; the caller
 *    (PyTorch's caching allocator on the Python side) owns every buffer; the library allocates nothing per call,
 *    never synchronises, and is CUDA-graph capturable; `stream` is a cudaStream_t passed as void*.
 *  - every function returns 0 on success, <0 on error; ddpm_last_error() returns the message (thread local).
 *    No exceptions or aborts cross the ABI (the reference raises Python exceptions: diffusion.py:42-43,119,133).
 *  - activations inside the engine are NHWC bf16; the 3-channel network input/output stay NCHW fp32 exactly
 *    as the reference hands them over (unet.py:205,232).
 */
#ifndef DDPM_B200_H
#define DDPM_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* ddpm_last_error(void);
/* 0 when the library was built for sm_100a and a CUDA driver + sm_100 device are present. */
int ddpm_runtime_check(void);
/* Device-side error flag set by a bounded wait that timed out inside a kernel (0 = none). Synchronises. */
int ddpm_device_error_flag(void);

/* Optional GroupNorm fusion of a conv / GEMM epilogue (nn.GroupNorm(32, C, eps=1e-6) of unet.py:18-20; csrc/gn_epilogue.cuh).
 *  qstats   the producer adds per (image, 4-channel quad) {sum, sum of squares} of its OUTPUT to qstats[NB][N/4][2]
 *           (fp64 atomics, caller zeroes it) - the statistics pass of the consuming GroupNorm disappears.  NULL = off. */
typedef struct ddpm_gn_epi {
    double* qstats;
} ddpm_gn_epi;

/* ------------------------------------------------------------------------------------------------
 * Low-level operator: one tcgen05 implicit-GEMM launch (used by the parity tests of the engine itself).
 * mode 0 (KK)   A K-major NHWC pixel tiles (+3x3 taps, up to 3 channel segments), B K-major matrix stack
 * mode 1 (MNMN) A,B MN-major, K over pixels (conv wgrad / P^T.dO); split-K with fp32 atomics
 * mode 2 (KMN)  A K-major, B MN-major (P.V)
 * replaces: F.conv2d (modules.py:121-123), F.linear (modules.py:59), torch.einsum x2 (unet.py:46-51) and their
 * autograd backward formulas.
 */
typedef struct ddpm_gemm_desc {
    int mode, block_n;                 /* block_n 0 = auto (64/128/256) */
    int M, N;                          /* output rows / cols per z slice */
    int W, H, NB;                      /* geometry of the NHWC tensors behind the 4-D maps (plain matrix: W=rows,H=1) */
    const void* a_ptr[3]; int a_C[3]; long long a_ld[3];   /* up to 3 A tensors: channels extent, pixel stride (elements) */
    int nseg; int seg_map[3], seg_taps[3], seg_kchunks[3], seg_cbase[3];
    const void* b_ptr; int b_K, b_rows, b_batch; long long b_ld, b_bs;  /* KK: [b_batch][b_rows][b_K]; MN modes: b_K = channel extent, b_ld = pixel stride */
    int b_k_base, a_z_n, b_z;
    int taps, splits, kblocks, a_c_base, b_c_base, grid_z;
    void* out; int ldo; long long out_z_stride, out_tap_stride; int flags;   /* flags: 1 = fp32 out, 2 = atomic add (fp32) */
    const float* bias; const float* rowvec; int rowvec_ld, rows_per_vec;
    const void* residual; int ldr; float alpha;
    /* stride-2 support: a_estride/b_estride = 2 builds the A (KK) / B (MNMN) map over a (W*2, H*2) tensor sampled with
     * elementStrides 2; seg_cmul multiplies the tile origin; seg_dx/seg_dy override the default 3x3 offsets when seg_custom != 0;
     * o_mul/o_py/o_px scatter output rows to pixel (y*o_mul+o_py, x*o_mul+o_px) of an (W*o_mul, H*o_mul) grid. */
    int a_estride, b_estride, b_pad;
    int seg_custom[3], seg_cmul[3]; signed char seg_dx[3][9], seg_dy[3][9];
    int o_mul, o_py, o_px;
    int kk_splits;                     /* mode 0: split the K loop over grid_z = kk_splits CTAs per tile (fp32 atomic output) */
    ddpm_gn_epi gn;                    /* mode 0 only, rows = NHWC pixels with H*W % 32 == 0 */
    int cta_pair;                      /* modes 0 / 1: 0 = library policy, 1 = single-CTA kernel, 2 = CTA-pair kernel (tcgen05 cta_group::2,
                                        * M = 256; error when the shape is not eligible), 3 = CTA-pair kernel when eligible */
} ddpm_gemm_desc;
int ddpm_gemm_run(const ddpm_gemm_desc* d, void* stream);

/* Low-level operator: 3x3 stride-1 convolution (+ optional fused 1x1 segments) with a haloed shared-memory input tile
 * (csrc/conv_halo.cuh) — the kernel behind ResidualBlock.conv1 / conv2(+skip) (unet.py:76,79,80) at resolutions >= 16x16.
 * a_ptr/a_C/a_ld: up to 3 NHWC bf16 inputs; segment s reads map seg_map[s] with seg_taps[s] in {9 (3x3, pad 1), 1 (1x1)},
 * seg_kchunks[s] chunks of 64 channels starting at channel seg_cbase[s]; w: packed bf16 [Cout][ldw], K order = segments,
 * then tap, then channel; out: NHWC bf16 [NB,H,W,Cout] = conv + bias + rowvec[image] + residual. */
typedef struct ddpm_halo_desc {
    int NB, H, W, Cout;
    const void* a_ptr[3]; int a_C[3]; long long a_ld[3];
    int nseg; int seg_map[3], seg_taps[3], seg_kchunks[3], seg_cbase[3];
    const void* w; long long ldw; int Ktot;
    void* out; const float* bias; const float* rowvec; int rowvec_ld; const void* residual;
    int base_offset_mode;              /* 0 = descriptor base_offset field left 0 (correct on B200); 1 = (addr>>7)&7 (probe) */
    int force_sub;                     /* 0 = auto; 1 / 2 = single-CTA kernel with that many 16x8 sub-tiles per CTA; 3 = CTA-pair kernel (cta_group::2) */
    ddpm_gn_epi gn;
    /* force_sub = 3 / CTA-pair kernel only: the 3x3 segment's input (map 0) is the RAW input of a GroupNorm(+SiLU); the kernel
     * applies y = act(sc*x + sh) to every landed tile in shared memory (unet.py:83-84: conv(act(norm(x)))), xf_K [NB][4][C] holding
     * {sc, sh, ...} per (image, channel).  NULL = off. */
    const float* xf_K; int xf_silu;
} ddpm_halo_desc;
int ddpm_conv_halo_run(const ddpm_halo_desc* d, void* stream);

/* Low-level operator: the attention core of AttentionBlock.forward (unet.py:43-51) as ONE kernel (csrc/attn_fused.cuh):
 * out[b] = softmax(Q K^T / sqrt(C)) V with q, k, v = the three C-channel thirds of qkv bf16 [NB][T][3C] (chunk order of unet.py:57),
 * out bf16 [NB][T][C].  S and O stay in tensor memory, P in shared memory.  Supported: T = 256 tokens (the 16x16 level), C = 256.
 * probs (optional, NULL = off): bf16 [NB][T][T], receives the softmax probabilities that the backward pass of a training plan
 * consumes (written from the shared-memory tile while P.V runs). */
int ddpm_attn_fused_run(const void* qkv, void* out, void* probs, int NB, int T, int C, void* stream);
/* Query-side half of the attention backward (autograd of unet.py:43-51) as ONE kernel: with P = probs saved by the forward,
 * dP = d_out V^T,  dS = P o (dP - rowsum(P o dP)) / sqrt(C)  -> d_scores bf16 [NB][T][T],  dQ = dS K -> the q third of
 * d_qkv bf16 [NB][T][3C].  dK = dS^T Q and dV = P^T d_out are plain GEMMs over d_scores / probs (ddpm_gemm_run).  T = 256, C = 256. */
int ddpm_attn_fused_bwd_run(const void* qkv, const void* d_out, const void* probs, void* d_scores, void* d_qkv, int NB, int T, int C, void* stream);

/* ------------------------------------------------------------------------------------------------
 * UNet engine.  replaces: UNet.__init__/forward (ddpm_torch/models/unet.py:96-233), its autograd backward,
 * and the model-side half of GaussianDiffusion.train_losses / p_sample_step (diffusion.py:107-158,217-243).
 */
typedef struct ddpm_unet_cfg {          /* mirrors UNet(in_channels, hid_channels, out_channels, ch_multipliers,   */
    int in_channels, hid_channels, out_channels;   /* num_res_blocks, apply_attn, time_embedding_dim, drop_rate)  unet.py:96-107 */
    /* in_channels / out_channels: 1..16 image channels (C*b*b of a block-size model); 5..16 need hid_channels % 64 == 0 and a
     * tensor-core resolution, otherwise ddpm_unet_workspace_bytes / ddpm_unet_plan return an error */
    int levels; int ch_mult[8];
    int num_res_blocks; int attn[8];
    int temb_dim;                       /* 0 -> 4*hid_channels (unet.py:112) */
    float drop_rate;
} ddpm_unet_cfg;
typedef struct ddpm_unet ddpm_unet;

int  ddpm_unet_create(const ddpm_unet_cfg* cfg, ddpm_unet** out);
void ddpm_unet_destroy(ddpm_unet* h);
/* Parameter inventory in the reference's state_dict order (unet.py registration order). Offsets (in fp32 elements)
 * address the FLAT parameter / gradient buffers the caller owns; each tensor is OIHW / [out,in] fp32 as in the reference. */
int       ddpm_unet_num_params(const ddpm_unet* h);
int       ddpm_unet_param_info(const ddpm_unet* h, int i, const char** name, int* ndim, int dims[4], long long* offset);
long long ddpm_unet_flat_elems(const ddpm_unet* h);
/* Workspace bytes for a (batch, H, W) plan; training != 0 also plans the backward pass. */
long long ddpm_unet_workspace_bytes(ddpm_unet* h, int B, int H, int W, int training);
/* Bind caller-owned device buffers and compile the launch plan. grads_flat may be NULL when training == 0. */
int ddpm_unet_plan(ddpm_unet* h, int B, int H, int W, int training, float* params_flat, float* grads_flat,
                   void* workspace, long long workspace_bytes);
/* Re-pack fp32 master weights into the bf16 kernel layouts; call after every parameter update / load_state_dict.
 * Ordered after everything queued on `stream` so far.  For a TRAINING plan the pack kernels run on the engine's internal stream
 * and the next forward/train_forward call joins them right before its first packed-weight consumer, so the pack overlaps the
 * timestep-embedding MLP and q_sample + in_conv of that forward; inference plans pack in `stream`. */
int ddpm_unet_repack(ddpm_unet* h, void* stream);
/* eps = UNet(x, t):  x f32[B,Cin,H,W] NCHW, t i64[B], eps f32[B,Cout,H,W]   (unet.py:205-233) */
int ddpm_unet_forward(ddpm_unet* h, const float* x, const int64_t* t, float* eps, uint64_t dropout_seed, void* stream);
/* Backward of the last forward: d_eps f32[B,Cout,H,W] -> flat grads (zeroed then written). x,t must be unchanged. */
int ddpm_unet_backward(ddpm_unet* h, const float* d_eps, void* stream);
/* Fused training forward (diffusion.py:217-243, mse/eps branch): x_t = q_sample(x0,t,noise) with the fp32 tables
 * tab_sqrt_ab / tab_sqrt_1mab [T]; eps = UNet(x_t,t); losses[b] = mean((noise-eps)^2). */
int ddpm_train_forward(ddpm_unet* h, const float* x0, const int64_t* t, const float* noise, const float* tab_sqrt_ab,
                       const float* tab_sqrt_1mab, float* losses, uint64_t dropout_seed, void* stream);
/* Backward of ddpm_train_forward given d(sum)/d(losses[b]) = gscale[b] (f32[B]). */
int ddpm_train_backward(ddpm_unet* h, const float* gscale, void* stream);
/* Sampler (diffusion.py:152-174, ddim.py:96-113).  setup uploads per-step tables: t_model[S] (timestep fed to the UNet),
 * coef[S][6] = {sqrt_recip_ab, sqrt_recip_m1_ab, post_c1, post_c2, exp(.5*logvar), t>0}; both HOST pointers.
 * reset(step) arms the device-side step counter; each step() call then consumes one step (counter decrements),
 * x f32[B,C,H,W] is updated in place; z = per-step N(0,1) draw (device) or NULL (+seed != 0: built-in Philox stream).
 * A step() is a fixed launch sequence with no host-side arguments that change -> capturable once, replayable T times.
 * The alpha/beta update runs in the epilogue of the UNet's final conv (eps never reaches memory; no tail launch). */
int ddpm_sampler_setup(ddpm_unet* h, int S, const int64_t* t_model_host, const float* coef_host);
int ddpm_sampler_reset(ddpm_unet* h, int first_step, void* stream);
int ddpm_sampler_step(ddpm_unet* h, float* x, const float* z, uint64_t seed, void* stream);
/* Same step, additionally writing the clipped x_0 prediction of diffusion.py:122,130 to pred_x0 f32[B,C,H,W] (NULL = skip):
 * GaussianDiffusion.p_sample_progressive (diffusion.py:176-198, p_sample_step(..., return_pred=True)). */
int ddpm_sampler_step_pred(ddpm_unet* h, float* x, const float* z, uint64_t seed, float* pred_x0, void* stream);
/* Data-parallel training (train.py:110 DDP, utils/train.py:149-153): the backward pass finishes the flat gradient buffer in
 * contiguous CHUNKS, level group by level group, and records a CUDA event per chunk.  grad_chunks returns their number and
 * fills lo/hi (element offsets into the flat buffer, in completion order; together they tile it exactly); wait_grad_chunk makes
 * `stream` wait for chunk i of the most recent ddpm_unet_backward / ddpm_train_backward, so that the caller can all-reduce that
 * chunk on a communication stream while the rest of the backward is still running.  Needs a training plan. */
int ddpm_unet_grad_chunks(const ddpm_unet* h, int max_n, long long* lo, long long* hi);
int ddpm_unet_wait_grad_chunk(ddpm_unet* h, int i, void* stream);
/* Introspection for tests / bench: op counts and algorithmic FLOPs of the compiled plan. */
int ddpm_unet_plan_stats(const ddpm_unet* h, int* n_fwd_ops, int* n_bwd_ops, int* n_tensorcore_ops, int* n_generic_ops,
                         double* fwd_flops, double* bwd_flops);
int ddpm_unet_launches_per_forward(const ddpm_unet* h);
/* kernel launches issued by one forward / backward / repack of the compiled plan (memsets not counted) */
int ddpm_unet_launch_counts(const ddpm_unet* h, int* fwd, int* bwd, int* pack);

/* ---- fused optimizer step over the flat fp32 buffers (SURVEY 8f rank 1).
 * Replaces, per training step, nn.utils.clip_grad_norm_(params, max_norm) + Adam.step() + LambdaLR warm-up + EMA.update()
 * (utils/train.py:159-165, :300-305; train.py:128-132) = ~13 tiny kernels x 304 tensors, by two launches and no host sync.
 *   step          : 1-based Adam step t (bias corrections 1 - beta^t), lr is the already-scheduled learning rate of this step
 *   max_grad_norm : <= 0 disables clipping;  ema_decay : < 0 disables the EMA update (ema_shadow may then be NULL);
 *   ema_num_updates: 0-based n of utils/train.py:301-302, decay_t = min(ema_decay, (1 + n) / (10 + n))
 *   state         : device scratch of >= 64 bytes, zero-initialised ONCE by the caller (fp64 accumulator + ticket)
 *   norm_out      : device float[2] <- {total_norm before clipping, clip coefficient applied}
 * n (elements) must be a multiple of 4 and all buffers 16-byte aligned (the flat layout guarantees both). */
typedef struct ddpm_opt_cfg {
  double lr, beta1, beta2, eps, max_grad_norm, ema_decay;
  int step, ema_num_updates;
} ddpm_opt_cfg;
int ddpm_opt_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* ema_shadow, long long n,
                  const ddpm_opt_cfg* cfg, void* state, float* norm_out, void* stream);

/* ---- generate.py:129 post-processing on the device (SURVEY 8f rank 3):
 * out[b][y][x][c] = uint8(clamp(round(x[b][c][y][x] * 127.5 + 127.5), 0, 255)) - NCHW fp32 samples -> NHWC uint8 images, the
 * layout PIL.Image.fromarray consumes (generate.py:112-114).  Bit-exact with the reference expression.  C in 1..4. */
int ddpm_to_uint8_nhwc(const float* x, uint8_t* out, int B, int C, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DDPM_B200_H */
