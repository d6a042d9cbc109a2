/* resshift_b200 — C ABI of the B200-native ResShift denoising hot path.
 *
 * The reference (zsyOAOA/ResShift) is pure Python/PyTorch and has no FFI; its plugin mechanism is
 * `instantiate_from_config` on yaml `target:` strings (reference utils/util_common.py:19-29, used at
 * sampler.py:87-88).  The entry points below are what a binding for the hot path needs; each cites the
 * reference interface it stands in for.  Conventions:
 *   - every function returns 0 on success, a negative code on failure; rs_last_error() gives the
 *     message (thread-local).  Nothing throws or exits across the boundary.
 *   - the CALLER owns all device memory (weight arena, workspace, inputs, outputs).  The library never
 *     allocates or frees device memory and never synchronises the device implicitly; all work is
 *     enqueued on the stream passed in (a cudaStream_t cast to void*), and is graph-capturable.
 *   - pointers are raw device pointers unless the name says `host`.  Tensors at the boundary are
 *     contiguous fp32 NCHW, exactly what the reference module receives/returns.
 *   - one host thread per engine (the reference is one single-threaded process per GPU, sampler.py:66-77).
 */
#ifndef RESSHIFT_B200_H
#define RESSHIFT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RS_MAX_LEVELS 8

/* Keyword arguments of UNetModelSwin.__init__ (reference models/unet.py:632-657) that shipped yaml
 * files vary.  Unsupported variants (dims != 2, resblock_updown, patch_norm, dropout > 0,
 * use_scale_shift_norm = False) are rejected by rs_unet_create. */
typedef struct rs_unet_config {
  int32_t image_size;
  int32_t in_channels;
  int32_t model_channels;
  int32_t out_channels;
  int32_t n_levels;
  int32_t channel_mult[RS_MAX_LEVELS];
  int32_t num_res_blocks[RS_MAX_LEVELS];
  int32_t n_attn;
  int32_t attention_resolutions[RS_MAX_LEVELS];
  int32_t swin_depth;
  int32_t swin_embed_dim;
  int32_t swin_heads;        /* swin_embed_dim / num_head_channels, or num_heads */
  int32_t window_size;
  float mlp_ratio;
  int32_t cond_mask;
  int32_t lq_size;
} rs_unet_config;

/* ``autoencoder.params`` of the shipped yaml files: VQModelTorch(ddconfig, n_embed, embed_dim)
 * (reference ldm/models/autoencoder.py:12-26; ddconfig -> ldm/modules/diffusionmodules/model.py:452-470,563-581).
 * Covered: double_z = False, attn_resolutions = [], dropout = 0 (every shipped config). */
typedef struct rs_vq_config {
  int32_t embed_dim;
  int32_t n_embed;
  int32_t z_channels;
  int32_t in_channels;
  int32_t out_ch;
  int32_t ch;
  int32_t n_levels;
  int32_t ch_mult[RS_MAX_LEVELS];
  int32_t num_res_blocks[RS_MAX_LEVELS];
} rs_vq_config;

typedef struct rs_engine rs_engine;     /* architecture + packed weights      */
typedef struct rs_plan rs_plan;         /* engine bound to (batch, H, W)      */
typedef struct rs_sampler rs_sampler;   /* plan + diffusion schedule (T steps) */

int rs_version(void);
const char* rs_last_error(void);

/* ---- denoiser: models.unet.UNetModelSwin (reference models/unet.py:603-912) ------------------ */
int rs_unet_create(const rs_unet_config* cfg, rs_engine** out);
void rs_unet_destroy(rs_engine* e);
/* state_dict inventory (reference key names / shapes; utils/util_net.py:86-98 relies on them) */
int rs_unet_param_count(const rs_engine* e);
int rs_unet_param_info(const rs_engine* e, int index, char* name, size_t name_cap, int32_t shape[4],
                       int32_t* ndim, int32_t* is_buffer);
/* packed (kernel-native, fp16/fp32) weight arena */
size_t rs_unet_arena_bytes(const rs_engine* e);
int rs_unet_set_arena(rs_engine* e, void* arena_dev);
/* repack one fp32 parameter (device pointer, reference layout: OIHW / [O, I] / [C]) into the arena */
int rs_unet_load_param(rs_engine* e, const char* name, const float* src_dev, void* stream);

/* ---- plan: the forward pass for a fixed (batch, latent H, latent W) -------------------------- */
int rs_plan_create(rs_engine* e, int batch, int height, int width, rs_plan** out);
void rs_plan_destroy(rs_plan* p);
size_t rs_plan_workspace_bytes(const rs_plan* p);
int rs_plan_bind(rs_plan* p, void* workspace_dev);   /* builds TMA descriptors; cheap, host only */
int rs_plan_num_launches(const rs_plan* p);          /* kernels per forward                       */
/* UNetModelSwin.forward(x, timesteps, lq=None, mask=None) (reference models/unet.py:865-895).
 * x [B, in_ch, H, W]; timesteps [B] (fp32); lq [B, 3, lq_h, lq_w]; mask [B, 1, lq_h, lq_w] or NULL;
 * out [B, out_ch, H, W].  All fp32 device pointers. */
int rs_plan_forward(rs_plan* p, const float* x, const float* timesteps, const float* lq, const float* mask,
                    float* out, void* stream);
/* measurement aid: one forward with CUDA events around every operator.  ms_by_kind[4] = conv/linear GEMM,
 * GroupNorm, window attention, upsample; conv_flops = algorithmic 2*MACs executed by the GEMM kernel. */
int rs_plan_profile(rs_plan* p, const float* x, const float* timesteps, const float* lq, const float* mask,
                    double* ms_by_kind, double* conv_flops, int32_t* n_conv_launches, void* stream);
/* per-operator variant: ms[i] and desc[i*desc_stride] for the first `cap` operators of the forward program */
int rs_plan_profile_ops(rs_plan* p, const float* x, const float* timesteps, const float* lq, const float* mask,
                        double* ms, char* desc, int desc_stride, int cap, int32_t* n_ops, void* stream);
/* debugging aid: copy an intermediate block output ("input_blocks.3", "middle_block", "output_blocks.11")
 * as fp32 NCHW into dst (device); returns channel count through *channels.  Valid right after a forward
 * only for blocks whose buffer is still live; used by the parity tests. */
int rs_plan_probe(rs_plan* p, const char* block, float* dst, int32_t* channels, int32_t* h, int32_t* w,
                  void* stream);

/* ---- sampler: SpacedDiffusion.p_sample_loop_progressive (reference models/gaussian_diffusion.py:421-472,
 *      p_sample :332-365, _scale_input :598-603, prior_sample :517-529; models/respace.py:43-63) ------ */
int rs_sampler_create(rs_plan* p, int steps, const double* sqrt_etas_host, double kappa,
                      const int32_t* timestep_map_host, rs_sampler** out);
void rs_sampler_destroy(rs_sampler* s);
/* z_y [B, C, H, W] fp32; noises [(T+1), B, C, H, W] fp32 in the reference's draw order (prior first);
 * lq/mask as in rs_plan_forward; out_latent [B, C, H, W] fp32 (the loop's final `sample`).
 * use_graph != 0 replays a CUDA graph captured on first use (same pointers required on later calls). */
int rs_sampler_run(rs_sampler* s, const float* z_y, const float* noises, const float* lq, const float* mask,
                   float* out_latent, int use_graph, void* stream);
/* Same call with HOST buffers (pinned or pageable): copies in, runs, copies the latent back, and
 * synchronises the stream.  This is the end-to-end entry the benchmark's `e2e` figure times. */
int rs_sampler_run_host(rs_sampler* s, const float* z_y_host, const float* noises_host, const float* lq_host,
                        const float* mask_host, float* out_latent_host, void* staging_dev, size_t staging_bytes,
                        int use_graph, void* stream);
size_t rs_sampler_staging_bytes(const rs_sampler* s);
/* optional taps for parity tests: per-step pred_xstart / sample, [T, B, C, H, W] fp32 device buffers or NULL */
int rs_sampler_set_taps(rs_sampler* s, float* pred_xstart_steps, float* sample_steps);

/* ---- VQ-GAN first stage: ldm.models.autoencoder.VQModelTorch (reference ldm/models/autoencoder.py:12-47) -------
 * The engine handle is the same opaque type as the denoiser's: rs_unet_param_count / _param_info / _arena_bytes /
 * _set_arena / _load_param work on it unchanged (state_dict names and shapes of the reference's VQModelTorch, so
 * autoencoder_vq_f4.pth / ffhq512_vq_f8_dim8_face.pth load as they are). */
int rs_vq_create(const rs_vq_config* cfg, rs_engine** out);
/* plan for a fixed (batch, image H, image W); which = 0: encode (image -> latent), 1: decode (latent -> image).
 * Uses rs_plan_workspace_bytes / rs_plan_bind / rs_plan_destroy like a denoiser plan. */
int rs_vq_plan_create(rs_engine* e, int batch, int image_h, int image_w, int which, rs_plan** out);
/* VQModelTorch.encode (autoencoder.py:28-31): x [B, 3, H, W] fp32 -> h [B, embed_dim, H/f, W/f] fp32 (f = 2^(levels-1)) */
int rs_vq_encode(rs_plan* p, const float* x, float* h_out, void* stream);
/* VQModelTorch.decode (autoencoder.py:33-40): h [B, embed_dim, H/f, W/f] -> quantize (VectorQuantizer2,
 * ldm/modules/vqvae/quantize.py:271-284; skipped when force_not_quantize) -> post_quant_conv -> Decoder -> [B, 3, H, W] fp32.
 * idx_out: optional [B, H/f, W/f] int32 code indices. */
int rs_vq_decode(rs_plan* p, const float* h, float* out, int32_t* idx_out, int force_not_quantize, void* stream);
/* diagnostics: per-launch times (ms) and descriptions of the plan's op list on the inputs of the last encode/decode
 * call (counterpart of rs_plan_profile_ops for the first-stage plans) */
int rs_vq_profile_ops(rs_plan* p, double* ms, char* desc, int desc_stride, int cap, int32_t* n_ops, void* stream);

/* ---- image edges of the sampler (reference sampler.py:176-223,286; utils/util_image.py:216-273,889-979) --------- */
/* F.interpolate(x, scale_factor=sf, mode='bicubic') on fp32 NCHW (models/gaussian_diffusion.py:503-504) */
int rs_op_bicubic_upsample(const float* x, int N, int C, int H, int W, int sf, float* y, void* stream);
/* uint8 HWC image(s) -> fp32 NCHW in [-1, 1]: (v / 255 - 0.5) / 0.5 */
int rs_op_ingest_u8(const void* src_u8_nhwc, int N, int H, int W, int C, float* dst_nchw, void* stream);
/* fp32 NCHW in [-1, 1] -> clamp, * 0.5 + 0.5, optional mask-back blend with lq (mask = 1 keeps the model output),
 * round(v * 255) -> uint8 HWC in RGB (bgr = 0) or BGR (bgr = 1) order (util_image.tensor2img) */
int rs_op_emit_u8(const float* sr_nchw, const float* lq_nchw_or_null, const float* mask_or_null, int N, int H, int W,
                  int bgr, void* dst_u8_nhwc, void* stream);
/* overlap-average of tiled results (ImageSpliterTh.update / gather): tiles [nty*ntx, N, C, th, tw] fp32 at output
 * origins ys[nty] / xs[ntx] (device int32 arrays) -> out [N, C, H, W] */
int rs_op_tile_gather(const float* tiles, int N, int C, int H, int W, int th, int tw, int nty, int ntx, const int32_t* ys,
                      const int32_t* xs, float* out, void* stream);

/* ---- single operators (unit tests / reuse) --------------------------------------------------- */
/* p_sample update (reference models/gaussian_diffusion.py:361-364 with :218-221) */
int rs_p_sample(const float* x_t, const float* x0_pred, const float* noise, float* x_next, float coef1,
                float coef2, float std, int t_is_zero, long long numel, void* stream);

/* conv / linear on NHWC fp16 views (reference nn.Conv2d / nn.Linear call sites, see csrc/conv_gemm.cuh).
 * x [N,H,W,C] with row stride ld; w_packed fp16 [Cout][k*k][Ipad] from rs_op_pack_conv_weight; optional
 * residual / fp16 output views (row strides res_ld / out_ld) and fp32 NCHW output; act 0 none, 1 GELU(erf),
 * 2 SiLU; bn = 0 lets the library choose the channel tile. */
int rs_op_pack_conv_weight(const float* src_oihw, void* dst_f16, int O, int I, int KH, int KW, int Ipad, void* stream);
int rs_op_conv2d(const void* x, int N, int H, int W, int C, int ld, const void* w_packed, int Ipad, const float* bias,
                 int Cout, int ksize, int stride, const void* residual, int res_ld, void* out, int out_ld,
                 float* out_f32_nchw, int act, int bn, void* stream);
/* conv2d + GroupNorm statistics of its output: part[N][slots][cstride][2] = (mean, M2) of the stored values per image /
 * 128-pixel tile slot / channel at channel offset coff; with gstat + counter (uint32[N], zeroed by the caller) the last
 * CTA of each image also writes gstat[N][32][2] = (group mean, group rstd) once slots * expected_channels channel-slots
 * arrived (expected_channels = 0: cstride).  reference: the GroupNorm32 that follows every conv (models/basic_ops.py:15-17) */
int rs_op_conv2d_stats(const void* x, int N, int H, int W, int C, int ld, const void* w_packed, int Ipad, const float* bias,
                       int Cout, int ksize, int stride, const void* residual, int res_ld, void* out, int out_ld, int act,
                       int bn, float* part, int cstride, int coff, int32_t* slots_out, float* gstat, void* counter,
                       int expected_channels, void* stream);
/* conv2d that may split its K loop over several CTAs (layers with few output tiles); scratch: 8*N*Ho*Wo*Cout floats */
int rs_op_conv2d_splitk(const void* x, int N, int H, int W, int C, int ld, const void* w_packed, int Ipad, const float* bias,
                        int Cout, int ksize, int stride, const void* residual, int res_ld, void* out, int out_ld, int act,
                        float* part, int cstride, int coff, float* scratch, int32_t* splits_out, float* gstat, void* counter,
                        void* stream);
/* profiling aid: `iters` launches of the same conv; per-CTA timeline of the last one in dbg (8 x u64 per CTA) */
int rs_op_conv2d_timeline(const void* x, int N, int H, int W, int C, int ld, const void* w_packed, int Ipad, const float* bias,
                          int Cout, int ksize, int stride, void* out, int out_ld, int bn, int iters, void* dbg,
                          int32_t* info, float* splitk_scratch_or_null, void* stream);
/* GroupNorm32 (+ FiLM scale/shift, + SiLU) (reference models/basic_ops.py:15-17, models/unet.py:198-202) */
int rs_op_groupnorm(const void* x, int N, int H, int W, int C, int ld, const float* gamma, const float* beta,
                    const float* film, long long film_sN, int silu, void* y, int y_ld, float* sums_scratch,
                    void* stream);
long long rs_op_groupnorm_scratch_floats(int N, int H, int W, int C);
/* the apply half alone, on gstat[N][32][2] = (group mean, group rstd) delivered by a producer (rs_op_conv2d_stats) */
int rs_op_groupnorm_apply(const void* x, int N, int H, int W, int C, int ld, const float* gamma, const float* beta,
                          const float* film, long long film_sN, int silu, void* y, int y_ld, const float* gstat,
                          void* stream);
/* ... or on the producers' raw (mean, M2) pairs part[N][slots][C][2]: the consumer combines them itself */
int rs_op_groupnorm_apply_pairs(const void* x, int N, int H, int W, int C, int ld, const float* gamma, const float* beta,
                                const float* film, long long film_sN, int silu, void* y, int y_ld, const float* part,
                                int slots, void* stream);
/* group statistics gstat[N][32][2] = (mean, rstd) from (mean, M2) pairs part[N][slots][C][2] (rows_per_slot values each)
 * as a kernel of its own — what the first-stage plans run in front of a GroupNorm whose producer has hundreds of tiles */
int rs_op_groupnorm_finalize(const float* part, int N, int slots, int C, int rows_per_slot, float eps, float* gstat, void* stream);
/* window attention core (reference models/swin_transformer.py:114-145,251-275); qkv [N,H,W,3*heads*32] */
int rs_op_expand_relpos(const float* table_225xh, float* dense_hx64x64, int heads, void* stream);
int rs_op_window_attention(const void* qkv, int N, int H, int W, int heads, int shift, const float* bias_dense,
                           void* out, void* stream);
/* fused attention half of a Swin block: y = x + proj(window_attention(qkv(norm1(x)))) (reference
 * models/swin_transformer.py:246-275 with WindowAttention.forward :114-145); x NHWC fp16 [N,H,W,E] (in place when
 * y == x), norm1 statistics as the producers' (mean, M2) pairs gn_part[N][gn_slots][E][2], weights packed fp16;
 * part_out (optional): pairs of y per 8x8 window, [N][(H/8)*(W/8)][E][2]; gstat_out (optional, tcgen05 kernel only, with
 * counters [N] zeroed by the caller): the 32 group (mean, rstd) of y per image, finalised by the last CTA to deliver
 * an image's pairs.  relbias_dense must be the output of
 * rs_op_expand_relpos (relative_position_bias_table gathered by relative_position_index, :82-97,130-133): the tcgen05
 * kernel keeps only its 225 distinct values per head (bias(i, j) depends on (yi - yj, xi - xj) alone).
 * RS_SWIN_IMPL=mma selects the mma.sync kernel (same arithmetic, reads the dense table as given). */
int rs_op_swin_attn(const void* x, int N, int H, int W, int E, int heads, int shift, const float* gn_part, int gn_slots,
                    const float* gamma, const float* beta, const void* wqkv_packed, const float* bqkv, const float* relbias_dense,
                    const void* wproj_packed, const float* bproj, void* y, float* part_out, float* gstat_out_or_null,
                    uint32_t* counters_or_null, void* stream);
/* fused single-head attention of the VQ-GAN bottleneck (reference AttnBlock.forward between the q / k / v convolutions
 * and proj_out, ldm/modules/diffusionmodules/model.py:180-203): per image n, out[n] = softmax(q[n] k[n]^T C^-1/2) v[n]
 * + v_bias with q, k [N][T][C] fp16, vt = v^T WITHOUT the bias [N][C][T] fp16, v_bias fp32 [C], out [N][T][C] fp16.
 * C a multiple of 64 in [64, 512], T a multiple of 64 (any size: the T x T scores never leave the chip). */
int rs_op_vq_attention(const void* q, const void* k, const void* vt, const float* v_bias, int N, int T, int C, void* out,
                       void* stream);
/* fused Swin MLP (reference models/swin_transformer.py:17-33,279): out = residual + fc2(GELU(fc1(x))) */
int rs_op_mlp(const void* x, int N, int H, int W, int E, int Hd, const void* w1_packed, const float* b1,
              const void* w2_packed, const float* b2, const void* residual, void* out, void* dbg_timeline_or_null,
              void* stream);
/* host-only: tile configuration the conv launcher picks: out[9] = BN, msub, stages, CTAs/SM, estimated cycles,
   CTAs per tile group (1 or 2), split-K factor, persistent kernel (0 / 1), cluster split-K (0 / 1) */
int rs_debug_tile_config(int m_tiles, int cout, int num_kblocks, int32_t* out);
/* profiling aid: later rs_op_swin_attn launches (tcgen05 kernel) write a clock64 timeline of CTA 0's first tile into
 * dev_buf[128 x int64] (two tiles x 64 stamps); NULL switches it off */
int rs_debug_swin_timeline(void* dev_buf_or_null);
/* nearest x2 (reference models/unet.py:71-81) */
int rs_op_upsample2x(const void* x, int N, int H, int W, int C, void* y, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RESSHIFT_B200_H */
