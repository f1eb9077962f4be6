/* libln3b200 -- C ABI of the B200-native LN3Diff generation hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b): every entry point takes a plain-C argument struct
 * of raw device pointers, explicit sizes/strides and enums, plus the CUDA stream as `void*`
 * (a cudaStream_t).  No torch types, no allocation, no retained pointers, no host
 * synchronisation: callers own every buffer (including workspaces).  All entry points return
 * LN3_OK (0) or a negative LN3_E* code; ln3_last_error() returns the thread-local message.
 * There is deliberately no CPU fallback: on a box without an sm_100 GPU every compute call
 * fails with LN3_ECUDA.
 *
 * Each entry point cites the reference code (NIRVANALAN/LN3Diff, paths relative to the
 * reference root) whose device work it replaces.  The reference has no FFI of its own -- it is
 * pure PyTorch -- so the "binding" is the ctypes stub in ln3diff_b200/_lib.py, mirrored for a
 * maintainer in INTEGRATION.md.
 */
#ifndef LN3B200_H_
#define LN3B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LN3_ABI_VERSION 1

#define LN3_OK 0
#define LN3_EINVAL (-1)       /* bad shape / alignment / enum */
#define LN3_ECUDA (-2)        /* CUDA runtime or driver error (includes: no GPU) */
#define LN3_EUNSUPPORTED (-3) /* configuration outside what the kernels implement */

int ln3_abi_version(void);
const char* ln3_last_error(void);
/* Number of kernels this library has launched in this process (for bench.py gpu_launches). */
unsigned long long ln3_launch_count(void);
/* A CUDA graph captured from these entry points re-executes its kernels without passing through
 * the library: callers add the graph's kernel-node count per replay to keep the tally honest. */
void ln3_add_launch_count(unsigned long long n);

/* ------------------------------------------------------------------ GEMM (tcgen05 + TMA)
 * out = epilogue(A[M,K] . W[N,K]^T): replaces every nn.Linear on the path
 *   dit/dit_models_xformers.py:231-323 (adaLN_modulation, FusedMLP), vit/vision_transformer.py:
 *   106-124 (qkv, proj), ldm/modules/attention.py:245-307 (to_q/k/v/out), dit/dit_decoder.py.
 * A, W bf16 row-major (K contiguous); fp32 accumulation in TMEM.
 * Epilogue: + bias[N] (fp32, optional) -> activation -> one of
 *   LN3_OUT_BF16       out bf16 [M, ldo]
 *   LN3_OUT_F32        out f32  [M, ldo]
 *   LN3_OUT_RESID_F32  out f32 residual stream updated in place:
 *                      out[m,n] += gate[(m / gate_rows) * gate_ld + n] * val   (gate NULL -> 1)
 *                      and, if out2 != NULL, out2 (bf16 [M, ldo2]) receives the updated row
 *                      (the un-normalised cross-attention query input of TextCondDiTBlock).
 * Constraints: K % 64 == 0, N % 128 == 0, 16-byte aligned pointers and leading dimensions.
 */
enum { LN3_ACT_NONE = 0, LN3_ACT_GELU_ERF = 1, LN3_ACT_GELU_TANH = 2, LN3_ACT_SILU = 3,
       LN3_ACT_QUICK_GELU = 4 /* x * sigmoid(1.702 x): the CLIP towers of the conditioners */ };
enum { LN3_OUT_BF16 = 0, LN3_OUT_F32 = 1, LN3_OUT_RESID_F32 = 2 };

typedef struct ln3_gemm_args {
  const void* A;   /* bf16 [M, lda] */
  const void* W;   /* bf16 [N, ldw] */
  const float* bias;
  void* out;
  void* out2;
  const float* gate;
  int M, N, K;
  long long lda, ldw, ldo, ldo2, gate_ld;
  int gate_rows;
  int act;
  int out_kind;
  /* optional per-head RMSNorm of the first head_norm_nsec column sections (each head_norm_sec_cols
   * wide, heads of 64 columns) before the bf16 store: y = x * rsqrt(mean_64(x^2) + eps) * w[sec][i].
   * This is `q, k = self.q_norm(q), self.k_norm(k)` (qk_norm=True, RMSNorm(64, eps 1e-5):
   * vit/vision_transformer.py:81-82,116; ldm/modules/attention.py:264-265,294) fused into the
   * projection GEMM.  head_norm_w: fp32 [head_norm_nsec, 64] or NULL.  LN3_OUT_BF16 only. */
  const float* head_norm_w;
  int head_norm_nsec;
  int head_norm_sec_cols;
  float head_norm_eps;
  /* optional scratch for the stream-K tail of the CTA-pair kernel: ln3_gemm_workspace_bytes() bytes of
   * device memory, 256-byte aligned, ZEROED ONCE by the caller (the kernel leaves it zeroed), never shared
   * by GEMMs that may run concurrently.  With T output tiles on P CTA pairs the last T % P tiles are split
   * along K over all pairs instead of leaving P - T % P pairs idle for a whole tile.  NULL -> plain tiles. */
  void* workspace;
  size_t workspace_bytes;
} ln3_gemm_args;

size_t ln3_gemm_workspace_bytes(void);

int ln3_gemm_bf16(const ln3_gemm_args* args, void* stream);

/* ------------------------------------------------------------------ attention (tcgen05)
 * out[b, i, h*64:(h+1)*64] = softmax(q_h k_h^T * scale) v_h, no mask: replaces
 * xformers.ops.memory_efficient_attention at vit/vision_transformer.py:114-118 (packed qkv of
 * MemEffAttention), ldm/modules/attention.py:279-307 (cross-attention, incl. its three
 * permute+contiguous copies) and the DiT2 decoder attention (dit/dit_decoder.py).
 * q/k/v/out are bf16; head h of row i of batch b lives at ptr + b*bs + i*ld + h*64, so a packed
 * (B, N, 3, H, 64) qkv buffer is addressed as q = base, k = base + H*64, v = base + 2*H*64 with
 * ld = 3*H*64.  Lq and Lkv are arbitrary (tails are zero-filled by TMA and masked).
 * head_dim must be 64 (every registry entry on the path except DiT-XL, SURVEY.md appendix A).
 */
typedef struct ln3_fmha_args {
  const void* q;
  const void* k;
  const void* v;
  void* out;
  int B, H, Lq, Lkv, head_dim;
  long long q_ld, q_bs, k_ld, k_bs, v_ld, v_bs, o_ld, o_bs; /* elements */
  float scale;
  /* optional second K/V source appended after the first along the sequence: the step-invariant DINO
   * tokens the I23D blocks concatenate to the latent tokens for self-attention
   * (dit/dit_models_xformers.py:522-530) -- their K/V are cached per prompt and never copied.
   * k2/v2 NULL -> unused. */
  const void* k2;
  const void* v2;
  int Lkv2;
  long long k2_ld, k2_bs, v2_ld, v2_bs;
  /* causal != 0: key j is visible to query i only when j <= i (the CLIP text tower of FrozenCLIPEmbedder,
   * sgm/modules/encoders/modules.py:347-408 -> transformers CLIPTextModel's causal mask); not with k2/v2. */
  int causal;
} ln3_fmha_args;

int ln3_fmha_fwd(const ln3_fmha_args* args, void* stream);

/* ------------------------------------------------------------------ norm + modulate (adaLN)
 * out_bf16[r, :] = norm(x[r, :]) * (1 + scale[g(r), :] (+ scale_tab)) + shift[g(r), :] (+ shift_tab)
 * with g(r) = r / mod_rows.  Replaces `modulate(self.norm1(x), shift, scale)` /
 * `t2i_modulate(...)` (dit/dit_models_xformers.py:47-53, 285-294, 518-530) and `modulate2` with
 * per-token operands (dit/dit_decoder.py:15-17; mod_rows = 1), producing the bf16 GEMM operand.
 *   norm = LN3_NORM_LAYER: LayerNorm without affine, biased variance, eps (1e-6 on the path)
 *          LN3_NORM_RMS  : x * rsqrt(mean(x^2) + eps) * weight        (dit/norm.py:27-40)
 *          LN3_NORM_NONE : identity (plain fp32 -> bf16 cast, optional activation LN3_ACT_*)
 * shift/scale NULL -> no modulation.  D must be a multiple of 128 and <= 2048.
 */
enum { LN3_NORM_NONE = 0, LN3_NORM_LAYER = 1, LN3_NORM_RMS = 2 };

/* OSG decoder arithmetic of the renderer / point queries */
enum { LN3_MLP_FP32 = 0, LN3_MLP_TF32 = 1 };

typedef struct ln3_norm_modulate_args {
  const float* x;     /* [rows, ldx]; updated in place when `resid` is given */
  void* out;          /* bf16 [rows, ldo] (NULL allowed with `resid`) */
  const float* shift; /* [groups, mod_ld] or NULL */
  const float* scale;
  const float* shift_tab; /* [D] or NULL: PixArt scale_shift_table rows */
  const float* scale_tab;
  const float* weight;    /* RMS weight [D] or NULL */
  int rows, D;
  long long ldx, ldo, mod_ld;
  int mod_rows;
  int norm;
  int act;            /* applied last (only with LN3_NORM_NONE) */
  float eps;
  /* optional fused residual update executed first, in place on x:
   *   x[r,:] += resid_gate[(r / resid_gate_rows), :] * resid[r,:]      (gate NULL -> 1)
   * i.e. the `x = x + gate * f(...)` of the DiT blocks (dit/dit_models_xformers.py:289-294,
   * 311-321) applied to the bf16 output of the preceding projection GEMM, so the residual stream is
   * read and written once, coalesced, by the kernel that normalises it anyway.  out may be NULL
   * (residual update only). */
  const void* resid;       /* bf16 [rows, resid_ld] or NULL */
  const float* resid_gate; /* fp32 [groups, resid_gate_ld] or NULL */
  long long resid_ld, resid_gate_ld;
  int resid_gate_rows;
  /* optional: rows outside [resid_row_begin, resid_row_end) take their residual from a per-group row
   *   resid_bcast[(r / resid_bcast_rows), :]   (bf16, row pitch resid_bcast_ld)
   * instead of resid[r,:] -- the cross-attention output of samples whose context tokens are all
   * identical (the zero-embedding unconditional half of classifier-free guidance,
   * sgm/modules/diffusionmodules/guiders.py:33-44 with force_uc_zero_embeddings): softmax over identical
   * keys is uniform, so the attention output is the one value row for every query.  NULL -> unused. */
  const void* resid_bcast;
  long long resid_bcast_ld;
  int resid_bcast_rows, resid_row_begin, resid_row_end;
  /* optional, with resid_bcast: the rows OUTSIDE [resid_row_begin, resid_row_end) additionally add their own
   * row of `resid` under a second gate,
   *   x[r,:] += resid_out_gate[(r / resid_out_gate_rows), :] * resid[r,:] + resid_bcast[...]
   * -- for those samples the preceding `x += gate_msa * attn` (dit/dit_models_xformers.py:311-312) has not been
   * applied yet: the pass that applies it exists only to produce the bf16 cross-attention query input, which the
   * closed-form samples do not need, so their self-attention and cross-attention residuals are applied together
   * here and the in-between pass covers the attended rows only.  NULL -> unused. */
  const float* resid_out_gate;
  long long resid_out_gate_ld;
  int resid_out_gate_rows;
} ln3_norm_modulate_args;

int ln3_norm_modulate(const ln3_norm_modulate_args* args, void* stream);

/* ------------------------------------------------------------------ timestep embedding
 * out_bf16[b, 0:128] = cos(t_b f_i), out[b, 128:256] = sin(t_b f_i), f_i = exp(-ln(1e4) i/128):
 * TimestepEmbedder.timestep_embedding (dit/dit_models_xformers.py:97-121), dim 256.
 */
int ln3_timestep_embedding(const float* t, int B, void* out_bf16, void* stream);

/* ------------------------------------------------------------------ patch embed (roll-out)
 * tokens[b, n*L + l, :] = Conv2d(k=s=2)(x[b, c*3+n, :, :])[l] + bias + pos_embed[n*L + l, :]
 * i.e. rearrange 'b (c n) h w -> (b n) c h w' + timm PatchEmbed + pos_embed
 * (dit/dit_trilatent.py:93-99).  x fp32 (B, 3*Cin, S, S) optionally pre-scaled per sample by
 * in_scale[b] (the denoiser's c_in, sgm/modules/diffusionmodules/denoiser.py:34-42);
 * weight fp32 (D, Cin, 2, 2); tokens fp32 (B, 3*(S/2)^2, D).
 */
typedef struct ln3_patch_embed_args {
  const float* x;
  const float* in_scale; /* [B] or NULL */
  const float* weight;
  const float* bias;
  const float* pos_embed; /* [3*L, D] or NULL */
  float* tokens;
  int B, Cin, S, D;
} ln3_patch_embed_args;

int ln3_patch_embed(const ln3_patch_embed_args* args, void* stream);

/* ------------------------------------------------------------------ final layer + unpatchify
 * FinalLayer / T2IFinalLayer (dit/dit_models_xformers.py:61-84, 655-678): LayerNorm(no affine,
 * eps 1e-6) -> modulate(shift, scale (+ tables)) -> Linear(D -> 4*Cout) -> unpatchify ->
 * '(b n) c h w -> b (c n) h w' (dit/dit_trilatent.py:130-140), fp32 contiguous output
 * (B, 3*Cout, S, S).  shift/scale are [B, mod_ld] rows.
 */
typedef struct ln3_final_layer_args {
  const float* x; /* tokens [B, 3*L, D] */
  const float* shift;
  const float* scale;
  const float* shift_tab;
  const float* scale_tab;
  const float* weight; /* [4*Cout, D] fp32 */
  const float* bias;   /* [4*Cout] */
  float* out;
  int B, S, D, Cout;
  long long mod_ld;
} ln3_final_layer_args;

int ln3_final_layer(const ln3_final_layer_args* args, void* stream);

/* ------------------------------------------------------------------ fused sampler update
 * x_out[b] = a[b] * x[b] + w0[b] * m0[b] + w1[b] * m1[b] + s[b] * noise[b]   (per-sample scalars)
 * One launch per step covering (SURVEY.md section 8a row S*):
 *   Euler-EDM + EpsScaling + VanillaCFG  sgm/modules/diffusionmodules/sampling.py:93-107,
 *       denoiser.py:25-42, guiders.py:24-31, sampling_utils.py:34-35  (m0 = uncond, m1 = cond)
 *   DDPM p_sample (eps/x0/v, fixed variance)  guided_diffusion/gaussian_diffusion.py:273-546
 *   flow-matching Euler + CFG              transport/integrators.py:101-120, dit/dit_i23d.py:155-168
 * coef is [B, 4] = (a, w0, w1, s); m1 / noise may be NULL when their weight is unused.
 */
typedef struct ln3_sampler_update_args {
  const float* x;
  const float* m0;
  const float* m1;
  const float* noise;
  const float* coef;
  float* x_out;
  int B;
  long long n_per_sample;
} ln3_sampler_update_args;

int ln3_sampler_affine_update(const ln3_sampler_update_args* args, void* stream);

/* ------------------------------------------------------------------ tri-plane volumetric renderer
 * ln3_render_views: the whole of ImportanceRenderer.forward (nsr/volumetric_rendering/renderer.py:
 * 133-307) for the Objaverse preset (nsr/script_util.py:761-797): 'auto' ray limits against the
 * box (math_utils.py:124-190, renderer.py:145-155), 64 stratified + 64 importance samples per ray,
 * tri-plane bilinear gather (renderer.py:55-104), in-box filter (:381-405), OSGDecoder
 * (nsr/triplane.py:339-375, FullyConnectedLayer gains nsr/networks_stylegan2.py:141-145),
 * MipRayMarcher2 (ray_marcher.py:26-68), sample_importance / sample_pdf (:479-552) and
 * unify_samples (:422-435), fused into one persistent warp-per-ray kernel.
 *
 *   planes_cl    fp32 [n_obj, 3, H, W, 32] channels-last (ln3_planes_to_channels_last)
 *   view_obj     int32 [V] object of each view, or NULL -> view v uses object v / views_per_obj
 *   ray_o, ray_d fp32 [V, M, 3]           (ln3_generate_rays, or caller supplied)
 *   noise_*      fp32 [V, M, 64] uniform [0,1): the tensors the reference draws with
 *                torch.rand_like (renderer.py:464) and torch.rand (renderer.py:530)
 *   w1,b1,w2,b2  raw OSGDecoder parameters (64,32), (64), (4,64), (4) -- gains applied inside
 *   rgb          fp32 [V, 3, M]  ('feature_samples' permuted: image_raw when reshaped to H x W)
 *   depth        fp32 [V, 1, M]   weights fp32 [V, 1, M]
 * group_size consecutive views share the reference's per-call global reductions (min/max of the
 * valid ray starts, depth clamp range): 1 when the reference renders one view per call
 * (nsr/train_util_diffusion.py:292-302), N for a batched Triplane.forward.
 * workspace: ln3_render_workspace_bytes(V, M, group_size) bytes of device memory.
 * dbg_* (optional, tests only): per-sample in-box masks [V*M,128] (coarse ++ fine), searchsorted
 * indices [V*M,64], sort permutation [V*M,128], fine depths [V*M,64].
 */
typedef struct ln3_render_args {
  const float* planes_cl;
  const int* view_obj;
  const float* ray_o;
  const float* ray_d;
  const float* noise_coarse;
  const float* noise_fine;
  const float* w1;
  const float* b1;
  const float* w2;
  const float* b2;
  float* rgb;
  float* depth;
  float* weights;
  void* workspace;
  size_t workspace_bytes;
  unsigned char* dbg_inbox;
  int* dbg_inds;
  int* dbg_order;
  float* dbg_zfine;
  int V, M, H, W, C, S, S_importance, hidden_dim, decoder_output_dim;
  int group_size, views_per_obj, white_back;
  int mlp_precision; /* LN3_MLP_FP32 (exact, SIMT) or LN3_MLP_TF32 (mma.sync tensor cores, fp32 accumulate) */
  double box_warp, bbox_min, bbox_max;
  /* optional: the M rays of a view are the pixels of an image of this width, m = y * image_w + x (RaySampler
   * order, ray_sampler.py:180-195).  When width and height are multiples of 4 the kernel walks 4x4 pixel tiles
   * (16 co-resident warps march through neighbouring texels in step: L1 reuse); 0 = plain ray order. */
  int image_w;
} ln3_render_args;

size_t ln3_render_workspace_bytes(int V, int M, int group_size);
int ln3_render_views(const ln3_render_args* args, void* stream);

/* ------------------------------------------------------------------ tri-plane point queries
 * ImportanceRenderer._run_model (nsr/volumetric_rendering/renderer.py:310-322) as driven by
 * forward_points / triplane_decode_grid (vit/vit_triplane.py:2009-2120) for mesh extraction:
 * sample_from_planes (bilinear, zeros padding, box_warp) + OSGDecoder at arbitrary points; no in-box
 * filter, no compositing.  sigma[n_obj][P] is the raw density logit, rgb[n_obj][P][3] the sigmoid
 * colour.  points == NULL -> the kernel generates the reference's grid itself (torch.linspace per axis
 * over [aabb_min, aabb_max], meshgrid 'ij'), P = grid_size^3: no 85 MB coordinate tensor, no
 * 2^16-point chunking, no empty_cache() between chunks.
 */
typedef struct ln3_query_points_args {
  const float* planes_cl; /* [n_obj][3][H][W][C] channels-last */
  const float* points;    /* [n_obj][P][3] or NULL (grid mode) */
  const float* w1;
  const float* b1;
  const float* w2;
  const float* b2;
  float* sigma;
  float* rgb;
  long long P;
  int n_obj, C, H, W, hidden_dim, decoder_output_dim, grid_size;
  int mlp_precision; /* LN3_MLP_FP32 or LN3_MLP_TF32 */
  float aabb_min_x, aabb_min_y, aabb_min_z, aabb_max_x, aabb_max_y, aabb_max_z;
  double box_warp;
} ln3_query_points_args;

int ln3_query_points(const ln3_query_points_args* args, void* stream);

/* RaySampler.forward (nsr/volumetric_rendering/ray_sampler.py:180-257): cams fp32 [V, 25]
 * (16 cam2world row-major + 9 intrinsics) -> ray_o, ray_d fp32 [V, res*res, 3], ray m = y*res + x. */
int ln3_generate_rays(const float* cams, int V, int res, float* ray_o, float* ray_d, void* stream);

/* (n_obj, 3*32, H, W) fp32 tri-plane as the VAE decoder emits it (vit/vit_triplane.py:1964,
 * channel = plane*32 + c) -> channels-last [n_obj, 3, H, W, 32] for the renderer's gathers. */
int ln3_planes_to_channels_last(const float* planes, int n_obj, int C, int H, int W, float* out,
                                void* stream);

/* ------------------------------------------------------------------ mesh extraction: marching cubes
 * Replaces the CPU `mcubes.marching_cubes(grid_out['sigma'] as (G,G,G) numpy, mesh_thres)` call of the mesh
 * export (nsr/train_util_diffusion.py:221-223; PyMCubes is an un-vendored third-party package) that follows
 * the G^3 point query (ln3_query_points).  grid fp32 [nx][ny][nz] (z fastest), exactly the array the reference
 * hands to mcubes.  Output is an indexed mesh like PyMCubes':
 *   vertices fp32 [n_vertices][3] = (i, j, k) index coordinates of the iso crossing on a lattice edge
 *            (linear interpolation, `value <= iso` classifies a corner), times scale[] plus offset[] per axis
 *            (scale 1 / offset 0 = mcubes; 2/(G-1)*0.45 and -0.45 fold the reference's :225-226 rescale in);
 *            ordered by (owning lattice point's linear index, axis)
 *   faces    int32 [n_faces][3] vertex indices, ordered by the cell's linear index; winding of the classic
 *            case table (normal towards the `<= iso` side), case tables generated by tools/gen_mc_tables.py.
 * Two calls because the sizes are data dependent: `_count` classifies and scans (totals[0] = n_vertices,
 * totals[1] = n_faces, device ints the caller reads back), `_emit` writes at most max_vertices / max_faces
 * entries.  workspace: ln3_marching_cubes_workspace_bytes(nx, ny, nz) bytes, 256-byte aligned, the SAME buffer
 * (contents preserved) for both calls. */
typedef struct ln3_marching_cubes_args {
  const float* grid;
  void* workspace;
  size_t workspace_bytes;
  int* totals;      /* device int[2] */
  float* vertices;  /* emit only */
  int* faces;       /* emit only */
  int nx, ny, nz;
  int max_vertices, max_faces;
  float iso;
  float scale[3];
  float offset[3];
} ln3_marching_cubes_args;

size_t ln3_marching_cubes_workspace_bytes(int nx, int ny, int nz);
int ln3_marching_cubes_count(const ln3_marching_cubes_args* args, void* stream);
int ln3_marching_cubes_emit(const ln3_marching_cubes_args* args, void* stream);

/* ------------------------------------------------------------------ frame sink
 * TrainLoopDiffusionWithRec.render_video_given_triplane's per-view host loop
 * (nsr/train_util_diffusion.py:292-376): `.cpu()` + numpy + matplotlib per view, replaced by one device
 * pass over all views so that one batched D2H copy (or the NCCL all-gather of frames) moves uint8.
 *   image  fp32 [N,3,H,W] in [-1,1] ('image_raw')
 *   depth  fp32 [N,1,H,W] ('image_depth') or NULL
 *   out    u8 [N, H, Wout, 3] (HWC video frames), Wout = W, or 2W with depth: [image | colour-mapped depth]
 * Arithmetic as the reference: byte = uint8(clip(v * 127.5 + 127.5, 0, 255)) (truncation), evaluated in float64
 * for the video frame with depth (the cat with the float64 colormap output promotes it, :340-345,366-368) and in
 * float32 (two rounded operations) for the image-only frame (the per-view image dump, :350-353);
 * depth -> (d - min_view) / (max_view - min_view) in fp32, colormap index min(trunc(x * 256), 255), the
 * byte table `lut` u8 [256,3] = uint8(clip((cmap_rgb * 2 - 1) * 127.5 + 127.5, 0, 255)) of the 256-entry
 * colormap (plt.cm.viridis in the reference); max == min gives the colormap's "bad" colour (0,0,0).
 * workspace: 2*N floats (per-view min / max).  W % 4 == 0. */
typedef struct ln3_pack_frames_args {
  const float* image;
  const float* depth;
  const unsigned char* lut;
  unsigned char* out;
  float* workspace;
  int N, H, W;
} ln3_pack_frames_args;

int ln3_pack_frames(const ln3_pack_frames_args* args, void* stream);

/* ------------------------------------------------------------------ VAE decoder: conv tail (NHWC fp32)
 * The reference's superresolution['conv_sr'] = ldm Decoder (ldm/modules/diffusionmodules/model.py:
 * 625-731) and PatchEmbedTriplane (vit/vit_triplane.py:58-108).  Activations are NHWC so the DiT2
 * token stream feeds conv_in directly and conv_out writes the renderer's channels-last tri-plane.
 *
 * ln3_conv_nhwc: out = conv(ksize in {1,3}, stride 1, pad ksize/2)(f(up(x))) + bias (+ residual)
 *   f = identity, or the fused GroupNorm-apply (+ swish): v*in_scale[n,c] + in_shift[n,c]
 *       (model.py:46-52 nonlinearity / Normalize; scale/shift from ln3_groupnorm_stats)
 *   up = identity or nearest 2x (Upsample, model.py:54-69): x is then [N, H/2, W/2, Cin]
 *   w is the Conv2d weight repacked to [ksize*ksize, Cin, Cout].
 * ln3_groupnorm_stats: torch.nn.GroupNorm(G, C, eps) statistics of x [N, HW, C] folded with the
 *   affine parameters into per-(image, channel) scale / shift [N, C].
 * ln3_attn_single_head: MemoryEfficientAttnBlock core (model.py:209-272): softmax(q k^T/sqrt(C)) v,
 *   q/k/v/out fp32 [N, L, C], one head of width C (128 in conv_sr).
 * ln3_patch_embed_triplane: Conv2d(3*Cz -> 3*E, k=s=2, groups=3) + the reference's
 *   (B,3E,h,w)->(B,E,3,h,w)->(B,3hw,E) reshape; x fp32 [B, 3*Cz, S, S] is pre-multiplied by in_mul
 *   (triplane_scaling_divider, nsr/train_util_diffusion.py:188); optional bf16 SiLU copy of the
 *   tokens (the adaLN operand of every DiT2 block, dit/dit_decoder.py:29-31).
 */
typedef struct ln3_conv_args {
  const float* x;
  const float* w;
  const float* bias;
  const float* in_scale;
  const float* in_shift;
  const float* residual;
  float* out;
  int N, H, W, Cin, Cout, ksize, upsample, in_swish;
  int precision; /* LN3_MLP_FP32 (exact SIMT) or LN3_MLP_TF32 (3x3 only: mma.sync tensor cores, fp32 accumulate) */
} ln3_conv_args;

int ln3_conv_nhwc(const ln3_conv_args* args, void* stream);
int ln3_groupnorm_stats(const float* x, const float* gamma, const float* beta, int N, int HW, int C,
                        int G, float eps, float* scale, float* shift, void* stream);
int ln3_attn_single_head(const float* q, const float* k, const float* v, float* out, int N, int L,
                         int C, void* stream);
int ln3_patch_embed_triplane(const float* x, const float* w, const float* bias, int B, int Cz, int S,
                             int E, float in_mul, float* tokens, void* silu_bf16, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LN3B200_H_ */
