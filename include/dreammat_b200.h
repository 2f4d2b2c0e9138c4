/*
 * dreammat_b200.h -- C-ABI of the B200-native DreamMat SDS inner loop.
 *
 * Drop-in boundary (SURVEY.md section 8b): every entry point replaces one native call the
 * reference's plugins make into an un-vendored CUDA dependency (nvdiffrast, tiny-cuda-nn,
 * _raytracing, envlight, diffusers/cuDNN).  The reference file:line each one stands in for
 * is cited beside it (paths relative to threestudio_dreammat/threestudio/).
 *
 * Conventions
 *   - all tensor pointers are DEVICE pointers unless the name ends in _host; row-major, dense;
 *   - `stream` is a cudaStream_t passed as void*;
 *   - return value: 0 on success, otherwise a cudaError_t (>0) or a DM_E* code (<0);
 *     dm_last_error() returns a static string for the calling thread;
 *   - no hidden allocations on the per-iteration entry points: scratch comes from the caller.
 */
#ifndef DREAMMAT_B200_H
#define DREAMMAT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DM_OK 0
#define DM_EINVAL (-1)
#define DM_EUNSUPPORTED (-2)
#define DM_EDRIVER (-3)

const char* dm_last_error(void);
int dm_version(void);
/* experiment knobs (no reference counterpart): "mc_skip_horizon" (0|1 skip below-horizon specular rays), "bvh_leaf" (1..4
 * triangles per BVH leaf, takes effect at the next dm_bvh_build), "pdl" (0|1 programmatic dependent launch of the dense kernels) */
int dm_tune(const char* key, int value);
int dm_tune_attention(int mode);       /* softmax variant: 0 fp32 exponentials, rescale every block (default, fastest measured);
                                      * 1 packed f16x2 exponentials + lazy rescale; 2 fp32 + lazy rescale */
/* split-K scratch: a caller-owned, ZERO-FILLED device buffer of fp32 partial sums (the finish kernel re-zeroes what it
 * reads, so it stays zero between calls).  Without a workspace split-K is not used.  One per process / device. */
/* pure query of the measured tile heuristic: kernel (0 single CTA, 1 CTA pair), tile width, split-K factor */
int dm_gemm_plan(int64_t M, int N, int K, int act, int bn_hint, int* kernel_out, int* bn_out, int* split_out);
size_t dm_gemm_workspace_bytes(void);
int dm_gemm_set_workspace(void* device_ptr, size_t bytes);
int dm_tune_gemm(int code);          /* 1|2: persistent CTAs per SM of the single-CTA kernel (tiles <= 128 wide);
                                      * 10|11|12: CTA-pair (cta_group::2) kernel off | heuristic | wherever possible;
                                      * 20|21: split-K of few-tile, long-K layers off | on;
                                      * 30|31|32: halo-reuse 3x3 convolution kernel (experiment) off | descriptor mode 1 | mode 2;
                                      * 40|41: two accumulators per tile in the single-CTA kernel (experiment) off | on */
/* number of kernels this library has launched in the process (bench.py's gpu_launches) */
long long dm_launch_count(void);
/* device sanity: returns 0 iff device `dev` is compute capability 10.x (sm_100a code present). */
int dm_device_check(int dev);

/* ------------------------------------------------------------------ geometry: hash grid + MLP
 * Replaces tcnn.Encoding (HashGrid) + VanillaMLP as called from
 * models/geometry/dreammat_mesh.py:239-254 via models/networks.py:55-64,150-187. */
typedef struct {
    int32_t n_levels;        /* 16 */
    int32_t n_features;      /* 2 (only value supported) */
    int32_t log2_hashmap;    /* 19 */
    int32_t base_resolution; /* 16 */
    float per_level_scale;   /* 1.447269237440378 */
    float bbox_min, bbox_max;/* contract_to_unisphere box: -radius, +radius (geometry/base.py:20-32) */
    int32_t n_hidden;        /* 64 */
    int32_t n_out;           /* 5 */
} dm_hashgrid_cfg;

/* host: total number of grid entries (x n_features = params); offsets_host gets n_levels+1 entry offsets */
int64_t dm_hashgrid_layout(const dm_hashgrid_cfg* cfg, uint32_t* offsets_host);
/* features[n,n_out] = MLP(HashGrid(contract(points[n,3]))) */
int dm_hashgrid_mlp_fwd(const dm_hashgrid_cfg* cfg, const float* points, int64_t n, const float* grid,
                        const float* W1, const float* W2, float* features, void* stream);
/* accumulates (+=) into dgrid, dW1, dW2; the forward is recomputed, nothing is saved */
int dm_hashgrid_mlp_bwd(const dm_hashgrid_cfg* cfg, const float* points, int64_t n, const float* grid,
                        const float* W1, const float* W2, const float* dfeatures, float* dgrid, float* dW1,
                        float* dW2, void* stream);
/* encoding only ([n, n_levels*n_features]); used by tests to pin the tcnn layout */
int dm_hashgrid_encode(const dm_hashgrid_cfg* cfg, const float* points, int64_t n, const float* grid, float* enc,
                       void* stream);

/* tangent-plane gaussian jitter, models/renderers/raytracing_renderer.py:161-173 */
int dm_jitter_positions(const float* pos, const float* nrm, const float* rand_ang, const float* normal_eps,
                        int64_t n, float* out, void* stream);

/* ------------------------------------------------------------------ BVH (replaces _raytracing)
 * models/renderers/raytracing_renderer.py:20-67 (RayTracer), :318-324 (miss <=> depth >= 10). */
typedef struct dm_bvh dm_bvh;
int dm_bvh_build(const float* verts_host, int64_t n_verts, const int32_t* tris_host, int64_t n_tris, dm_bvh** out);
void dm_bvh_free(dm_bvh* bvh);
int64_t dm_bvh_num_nodes(const dm_bvh* bvh);
/* closest hit: t[n] (10.0 on miss), tri[n] (-1 on miss), uv[n,2] (barycentrics of vertex 1, 2); uv may be NULL */
int dm_bvh_trace(const dm_bvh* bvh, const float* rays_o, const float* rays_d, int64_t n, float* t, int32_t* tri,
                 float* uv, void* stream);

/* ------------------------------------------------------------------ G-buffer (replaces dr.rasterize + dr.interpolate)
 * models/renderers/raytracing_renderer.py:122-159, utils/rasterize.py:22-78.  Visibility at
 * pixel centres by closest hit of the pixel-centre ray; outputs in nvdiffrast's layout.
 * v_pos/v_nrm [V,3], tris [F,3] int32 (device); rays_o/rays_d [B,H,W,3]; mvp,w2c [B,4,4].
 * rast [B,H,W,4] = (u,v,z/w,tri_id+1); gb_pos/gb_nrm [B,H*W,3]; mask [B,H*W] uint8;
 * comp_normal [B,H,W,3] (view-space normal map over bg (.5,.5,1), no antialias). */
int dm_raster_gbuffer(const dm_bvh* bvh, const float* v_pos, const float* v_nrm, const int32_t* tris,
                      const float* rays_o, const float* rays_d, const float* mvp, const float* w2c, int B, int H,
                      int W, float* rast, float* gb_pos, float* gb_nrm, uint8_t* mask, float* comp_normal,
                      void* stream);
/* row-major stream compaction of mask -> pixel indices; count_host receives pn.  (init-time; syncs) */
int dm_compact_mask(const uint8_t* mask, int64_t n, int32_t* idx_out, int64_t* count_host, void* stream);
/* dst[i,:] = src[idx[i],:] for c floats per row */
int dm_gather_rows(const float* src, const int32_t* idx, int64_t n, int c, float* dst, void* stream);
/* depth map, raytracing_renderer.py:129-134: per-batch min/max of 1/(z/w + 1e-6) over mask, -> [0.3,1] */
int dm_depth_normalize(const float* rast, const uint8_t* mask, int64_t n_pix, float* depth_out, float* scratch2,
                       void* stream);

/* ------------------------------------------------------------------ material (a4/a5)
 * models/materials/dreammat_material.py:713-763 */
typedef struct {
    float min_metallic, max_metallic;       /* 0.0, 0.9 */
    float min_roughness, max_roughness;     /* MC: 0.01, 0.9 (roughness^2); split-sum: 0.1, 0.95 */
    int32_t n_diffuse, n_specular;          /* 200, 128 */
} dm_material_cfg;

/* Monte-Carlo shading, dreammat_material.py:615-677 (+ :490-507 get_lights, :439-455 env lookup,
 * :554-596 sampling).  env_rgba: [envH,envW] float4 (rgb + pad) built by dm_envmap_pack.
 * tab_d [n_diffuse,2], tab_s [n_specular,2]: the (ua,ue) tables of :389-398.
 * rand_d, rand_s [n]: uniform draws (:567, :590).
 * Outputs: color [n,3] (sRGB, differentiable), jac [n,9] = d color_c / d (albedo_c, metallic, a)
 * for c=0..2, reg_sums[2] += (sum luma*|dkd_b|, sum |dks0|*|dks1|); aux pointers may be NULL:
 * albedo[n,3] roughness[n] metalness[n] spec_light[n,3] diff_light[n,3] spec_color[n,3] diff_color[n,3].
 * hit_bits (optional, zero-initialised by the caller): [n, ceil((nd+ns)/32)] occlusion bit per sample id.
 * sample_perm (optional): visiting order of the sample ids (a permutation of 0..nd-1 followed by one of
 * nd..nd+ns-1); sums are order-independent, a direction-coherent order cuts BVH traversal divergence. */
int dm_shade_mc_fwd(const dm_material_cfg* cfg, const dm_bvh* bvh, const float* env_rgba, int envH, int envW,
                    const float* tab_d, const float* tab_s, const float* pts, const float* normals,
                    const float* viewdirs, const float* features, const float* features_jitter,
                    const float* rand_d, const float* rand_s, int64_t n, float* color, float* jac,
                    float* reg_sums, float* albedo, float* roughness, float* metalness, float* spec_light,
                    float* diff_light, float* spec_color, float* diff_color, uint32_t* hit_bits,
                    const int32_t* sample_perm, void* stream);

/* Split-sum shading, dreammat_material.py:679-711.  fg_lut [256,256,2]; diffuse_cube [6,rd,rd,3];
 * spec_mips: n_mips device pointers (host array) to [6,r_i,r_i,3], r_i = spec_res0 >> i. */
int dm_shade_splitsum_fwd(const dm_material_cfg* cfg, const float* fg_lut, int lut_res, const float* diffuse_cube,
                          int diff_res, const float* const* spec_mips_host, int n_mips, int spec_res0,
                          const float* normals, const float* viewdirs, const float* features,
                          const float* features_jitter, int64_t n, float* color, float* jac, float* reg_sums,
                          float* albedo, float* roughness, float* metalness, float* spec_light, float* diff_light,
                          float* spec_color, float* diff_color, void* stream);

/* backward of either shading path: dfeatures[n,5], dfeatures_jitter[n,5] (overwritten).
 * dcolor [n,3]; reg_scale = d loss / d mat_reg_sum terms: dreg_kd = lambda*0.25/n_total, dreg_ks = lambda*0.1/n_total */
int dm_shade_bwd(const dm_material_cfg* cfg, const float* features, const float* features_jitter,
                 const float* dcolor, const float* jac, float dreg_kd, float dreg_ks, int64_t n, float* dfeatures,
                 float* dfeatures_jitter, void* stream);

/* [H,W,3] float -> [H,W] float4 */
int dm_envmap_pack(const float* rgb, int64_t n_texels, float* rgba, void* stream);

/* ------------------------------------------------------------------ canvas (a6)
 * raytracing_renderer.py:189-207 without the antialias pass: canvas = 1; canvas[pix[i]] = color[i]. */
int dm_scatter_canvas(const float* values, const int32_t* pix, int64_t n, int c, float* canvas, void* stream);
int dm_fill(float* p, int64_t n, float v, void* stream);
/* dvalues[i,:] = dcanvas[pix[i],:] */
int dm_gather_canvas_grad(const float* dcanvas, const int32_t* pix, int64_t n, int c, float* dvalues, void* stream);

/* silhouette antialias (dr.antialias, utils/rasterize.py:56 <- raytracing_renderer.py:127,147,199) as a sparse
 * blend whose pair list (dst pixel, src pixel, weight) is fixed per view and built once on the host
 * (dreammat_b200/antialias.py): out = in; out[dst[k]] += alpha[k] * (in[src[k]] - in[dst[k]]).  bwd is its adjoint. */
int dm_antialias_fwd(const float* in, const int32_t* dst, const int32_t* src, const float* alpha, int64_t k,
                     int64_t n_pix, int c, float* out, void* stream);
int dm_antialias_bwd(const float* dout, const int32_t* dst, const int32_t* src, const float* alpha, int64_t k,
                     int64_t n_pix, int c, float* din, void* stream);

/* F.interpolate(rgb, (512,512), mode="bilinear", align_corners=False) before the VAE when the render is not 512^2
 * (dreammat_guidance.py:507-513), NHWC fp32.  adjoint=0: in [n,Hi,Wi,c] -> out [n,Ho,Wo,c]; adjoint=1: in is
 * d out [n,Ho,Wo,c] and out receives d in [n,Hi,Wi,c]. */
int dm_resize_bilinear(const float* in, int n, int Hi, int Wi, int Ho, int Wo, int c, float* out, int adjoint,
                       void* stream);

/* ------------------------------------------------------------------ optimiser (a9)
 * torch.optim.Adam as configured by systems/utils.py:34-53 + configs/dreammat.yaml:110-115 */
int dm_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                 float eps, int32_t step, float grad_scale, void* stream);

/* ------------------------------------------------------------------ CSD / SDS combine (a8 tail, a9)
 * models/guidance/dreammat_guidance.py:475-481,584-594.
 * eps_pred [3,B,C,H,W] (text, uncond, null) fp32; noise, latents [B,C,H,W]; w[B] = 1 - alphas_cumprod[t].
 * grad = nan_to_num(w*(c*e_text + u*e_uncond + nl*e_null + s*noise)); dlatents = grad / B;
 * norms[10]: loss_sds, grad_norm, uncond_m_noise, text_m_noise, text_m_uncond, text_m_null,
 * null_m_uncond, noise, uncond, text (squared sums; sqrt taken by the host). */
int dm_sds_grad(const float* eps_pred, const float* noise, const float* w, int B, int64_t chw, float c_text,
                float c_uncond, float c_null, float c_noise, float* grad, float* dlatents, float* norms,
                void* stream);

/* ------------------------------------------------------------------ split-sum environment lights (a5 / N4)
 * Device-side build of `envlight.EnvLight(path, scale)` (ashawkey/envlight wrapping nvdiffrec renderutils, un-vendored;
 * models/materials/dreammat_material.py:379-386): lat-long HDR [H,W,3] * scale -> cube [6,res,res,3]; 2x2-average mips;
 * mode 0 cosine (diffuse) / mode 1 GGX-prefiltered (specular, alpha^2 = roughness^4, texels with N.L >= cos_cutoff)
 * convolution at equal resolution.  Host driver + disk cache: dreammat_b200/envlight.py. */
int dm_envlight_latlong_to_cube(const float* latlong, int H, int W, float scale, int res, float* cube, void* stream);
int dm_envlight_downsample(const float* cube, int res, float* out, void* stream);
int dm_envlight_filter(const float* cube, int res, int mode, float roughness, float cos_cutoff, float* out, void* stream);

/* ------------------------------------------------------------------ dense path (a7, a8)
 * Tensor-core (tcgen05 + TMA + TMEM) contraction used for every conv / linear of the VAE encoder,
 * UNet and ControlNet: replaces the cuDNN / cuBLAS kernels diffusers dispatches from
 * models/guidance/dreammat_guidance.py:218-229, :274-282, :290.  fp16 (bf16=0) or bf16 operands,
 * fp32 accumulation.  Epilogue order: acc*alpha + bias + rowvec -> act -> + residual -> * out_scale. */
typedef struct {
    const void* bias;          /* [N] or NULL */
    const void* rowvec;        /* [M / rows_per_vec, N] (per-image vector, e.g. time embedding) or NULL */
    int32_t rows_per_vec;
    int32_t ld_rowvec;
    const void* residual;      /* [M, ld_res] or NULL */
    int32_t ld_res;
    int64_t res_batch_stride;
    float alpha;
    float out_scale;
    int32_t act;               /* 0 none, 1 SiLU, 2 GELU(erf), 3 GEGLU: B rows interleaved [32 value | 32 gate],
                                * C gets N/2 columns value*gelu(gate) (attention.py GEGLU of the FF block) */
    int32_t out_f32;           /* 1: C is float32 */
} dm_epilogue;

/* C[b] = epi(A[b] . B[b]^T): A [M,K] row stride lda, B [N,K] row stride ldb (K-major both), K % 64 == 0.
 * b_batch_stride == 0 shares B across the batch. */
int dm_gemm(int bf16, const void* A, int64_t lda, int64_t a_batch_stride, const void* B, int64_t ldb,
            int64_t b_batch_stride, void* C, int64_t ldc, int64_t c_batch_stride, int M, int N, int K, int batch,
            const dm_epilogue* ep, int bn_hint, void* stream);
/* NHWC implicit-GEMM convolution: x [n,H,W,Cin] (Cin % 64 == 0), w [Cout, k*k*Cin] (tap-major, channel
 * minor), y [n,Ho,Wo,ldc]; zero padding pad_t/pad_l at the top/left, implicit at the bottom/right. */
int dm_conv2d(int bf16, const void* x, int n_img, int H, int W, int Cin, const void* w, int Cout, int ksize,
              int stride, int pad_t, int pad_l, int Ho, int Wo, void* y, int64_t ldc, const dm_epilogue* ep,
              int bn_hint, void* stream);

/* conv_out of the UNet with the CSD / SDS combination fused into its epilogue: the model-level tail of
 * `dm_unet_fwd_sds` (SURVEY.md section 8b).  Replaces conv_out (dreammat_guidance.py:274-282), the `.sample` layout /
 * dtype change and compute_grad_sds' tail + nan_to_num + the logged norms (:475-495, :584-594) by one kernel: a CTA
 * computes the three CFG-branch tiles of the same 128 latent pixels back to back and combines them in registers.
 * x [3B, H, W, Cin] NHWC ordered [branch: text | uncond | null][view]; w [4, 9*Cin]; bias [4] (storage dtype).
 * noise [B,4,H*W] fp32, w1mac[B] = 1 - alphas_cumprod[t]; coef (DEVICE, so a captured graph can be replayed with new
 * schedule values) = {c_text, c_uncond, c_null, c_noise, dlat_scale}.  Outputs (NCHW fp32): grad, dlatents = grad *
 * dlat_scale (either may be NULL), norms[10] += the squared sums listed at dm_sds_grad, eps_out [3,B,4,H*W] optional. */
typedef struct {
    const float* noise;
    const float* w;
    const float* coef;
    float* grad;
    float* dlatents;
    float* norms;
    float* eps_out;
} dm_csd;
int dm_conv2d_csd(int bf16, const void* x, int B, int H, int W, int Cin, const void* w, const void* bias, const dm_csd* c,
                  void* stream);

/* ---- high-precision mode (half_precision_weights=false, models/guidance/dreammat_guidance.py:56,92-94) ----
 * fp32 storage end to end.  The contractions still run on the bf16 tcgen05 kernel: both operands are split into three
 * bf16 terms (24 mantissa bits) and the six significant partial products are laid side by side along K,
 *     A' = [a1|a2|a1|a3|a2|a1],  B' = [b1|b1|b2|b1|b2|b3]   (K' = 6K; for a conv: 6*Cin channels per tap),
 * so dm_gemm / dm_conv2d(bf16=1, out_f32=1, no epilogue terms) return A.B^T to fp32 accuracy; dm_hp_epilogue then
 * applies the dm_epilogue terms (all pointers fp32) to the raw accumulators.  Every streaming entry point below
 * accepts 2 as its `bf16` selector = fp32 storage.
 * dm_hp_split: x [rows, ldx] (first `cols` columns) fp32 -> out [rows, 6*cols] bf16; pattern 0 = A operand, 1 = B operand
 * (conv weights [Cout, taps*Cin]: rows = Cout*taps, cols = Cin). */
int dm_hp_split(const float* x, int64_t rows, int cols, int64_t ldx, int pattern, void* out_bf16, void* stream);
/* raw [rows, N] fp32 accumulators -> out (row stride ldc, batch stride out_batch_stride, rows_per_batch rows per batch):
 * acc*alpha + bias + rowvec -> act -> + residual -> * out_scale; act 3 (GEGLU) writes N/2 columns */
int dm_hp_epilogue(const float* raw, int64_t rows, int N, int64_t rows_per_batch, const dm_epilogue* ep, float* out,
                   int64_t ldc, int64_t out_batch_stride, void* stream);

/* ---- streaming kernels of the dense path (NHWC; storage selected by `bf16`: 0 fp16, 1 bf16, 2 fp32; fp32 math) ---- */
/* torch.nn.GroupNorm (+ optional SiLU) as used by diffusers ResnetBlock2D / Transformer2DModel.norm.
 * x [n_img, HW, ld] (first C channels), y [n_img, HW, ldy]; stats [n_img*G*2] receives (sum, sumsq)
 * per group and is what dm_groupnorm_bwd needs. */
int dm_groupnorm(int bf16, const void* x, int n_img, int HW, int C, int ld, int G, const void* gamma,
                 const void* beta, float eps, int silu, void* y, int ldy, float* stats, void* stream);
/* dx = d/dx [ act(GN(x)) ] . dz (+ dx_add); x, dz, dx dense [n_img, HW, C]; bstats scratch [n_img*G*2] */
int dm_groupnorm_bwd(int bf16, const void* x, const void* dz, int n_img, int HW, int C, int G, const void* gamma,
                     const void* beta, float eps, int silu, const float* stats, float* bstats, const void* dx_add,
                     void* dx, void* stream);
int dm_layernorm(int bf16, const void* x, int64_t M, int C, const void* gamma, const void* beta, float eps, void* y,
                 void* stream);
/* out[m,j] = h[m,j] * gelu(h[m,D+j]), h [M,2D] */
int dm_geglu(int bf16, const void* h, int64_t M, int D, void* out, void* stream);
/* nearest 2x (zero_insert=0) or zero-insertion 2x (zero_insert=1, adjoint of a stride-2 gather) */
int dm_upsample2x(int bf16, const void* x, int n, int H, int W, int C, int zero_insert, void* y, void* stream);
/* dst[r,0:cols] = a*s1[r,0:cols] + b*s2[r,0:cols] (s2 may be NULL) with independent row strides */
int dm_axpby2d(int bf16, const void* s1, int64_t ld1, float a, const void* s2, int64_t ld2, float b, int64_t rows,
               int cols, void* dst, int64_t ldd, void* stream);
int dm_transpose(int bf16, const void* x, int batch, int R, int C, int64_t ldx, int64_t bsx, void* y, int64_t ldy,
                 int64_t bsy, void* stream);
int dm_softmax_rows(int bf16, const void* x, int64_t rows, int cols, int64_t ld, float scale, void* y, void* stream);
int dm_softmax_bwd(int bf16, const void* P, const void* dP, int64_t rows, int cols, int64_t ld, float scale, void* dS,
                   void* stream);
/* fp32 [rows,cin] -> T [rows,cpad] (x*scale+shift, zero padding) and back (first cout channels, * scale) */
int dm_pad_convert(int bf16, const float* x, int64_t rows, int cin, int cpad, float scale, float shift, void* y,
                   void* stream);
/* N1: gather + de-quantise the resident pre-rendered condition maps (data/uncond.py:532-582,799-802) straight into the
 * channel-padded ControlNet condition [B, HW, cpad] (storage dtype): depth fp32 [V,HW] | normal u8 [V,HW,3] / 255 |
 * light u8 [V,E,HW,18] / 255 for the batch's (view_ids[b], env_ids[b]); the fp32 condition_map never exists. */
int dm_cond_gather(int bf16, const float* depth, const uint8_t* normal, const uint8_t* light, int n_env, int64_t HW,
                   const int32_t* view_ids, const int32_t* env_ids, int B, int cpad, void* out, void* stream);
int dm_unpad_convert(int bf16, const void* x, int64_t rows, int ld, int cout, float scale, float* y, void* stream);
int dm_nhwc_to_nchw_f32(int bf16, const void* x, int n, int HW, int ld, int C, float* y, void* stream);
/* DiagonalGaussianDistribution.sample() * scaling_factor (dreammat_guidance.py:290-291) and its backward */
int dm_vae_sample(int bf16, const void* moments, int n, int HW, int ld, const float* eps, float scaling, float* z,
                  void* stream);
int dm_vae_sample_bwd(int bf16, const void* moments, int n, int HW, int ld, const float* eps, float scaling,
                      const float* dz, void* dmoments, void* stream);
/* scheduler.add_noise + CFG replication (dreammat_guidance.py:463, :407): out [rep*B, HW, cpad] */
int dm_add_noise(int bf16, const float* z, const float* noise, const float* sqrt_ac, const float* sqrt_1mac, int B,
                 int HW, int cpad, int rep, void* out, void* stream);
int dm_timestep_embedding(int bf16, const float* t, int n, int dim, void* out, void* stream);
int dm_silu(int bf16, const void* x, int64_t n, void* y, void* stream);

/* Fused attention, head_dim 64: O = softmax(scale * Q K^T) V per (batch, head).  Q [batch,Nq,ldq],
 * K/V [batch,Nk,ldkv], O [batch,Nq,ldo]; head h occupies columns [64h, 64h+64) of every operand.
 * Replaces SDPA in diffusers' BasicTransformerBlock (self- and cross-attention). */
int dm_attention(int bf16, const void* q, int64_t ldq, int64_t q_batch_stride, const void* k, const void* v,
                 int64_t ldkv, int64_t kv_batch_stride, void* out, int64_t ldo, int64_t out_batch_stride, int batch,
                 int heads, int Nq, int Nk, int head_dim, float scale, void* stream);

/* ------------------------------------------------------------------ texture bake of the mesh exporter (N5)
 * Replaces the texture half of threestudio's `mesh-exporter` (models/exporters/mesh_exporter.py: nvdiffrast UV
 * rasterisation, per-texel geometry/material export, cv2.inpaint seam padding).  The UV atlas comes from
 * dreammat_b200/uvatlas.py.  T (texture size) must lie in [16, 8192].  Init-time entry points; bit-reproducible.
 * dm_uv_raster: uv_fixed [Vt,2] int32 texel coordinates with 8 sub-texel bits, tri_uv [F,3]; texel (r,c) has its centre at
 *   (256c+128, 256r+128).  int64 edge functions + top-left rule; faces whose snapped area is <= 0 cover nothing.  The
 *   caller guarantees that no texel centre is covered twice (the atlas is checked for it).
 *   owner [T*T] face id or -1; bary [T*T,3] fp32 barycentrics; mask [T*T] 1 where covered. */
int dm_uv_raster(const int32_t* uv_fixed, const int32_t* tri_uv, int64_t n_faces, int T, int32_t* owner, float* bary,
                 uint8_t* mask, void* stream);
/* points[i] = sum_k bary[texels[i],k] * v_pos[t_pos_idx[owner[texels[i]], k]]  (texels: from dm_compact_mask of mask) */
int dm_texel_positions(const int32_t* texels, int64_t n, const int32_t* owner, const float* bary, const float* v_pos,
                       const int32_t* t_pos_idx, float* points, void* stream);
/* DreamMatMaterial.export (dreammat_material.py:765-797) of features [n,5]: sigmoid; metallic range; roughness
 * sqrt(m*(max-min)+min+1e-7) with cfg->min_roughness / max_roughness holding the SQUARED-roughness range.
 * out [n,5] (albedo rgb, metallic, roughness; may be NULL); texels (may be NULL): scatter (uint8)(x*255) into
 * map_kd [T*T,3], map_pm [T*T], map_pr [T*T] at texels[i]. */
int dm_material_export(const dm_material_cfg* cfg, const float* features, int64_t n, float* out, const int32_t* texels,
                       uint8_t* map_kd, uint8_t* map_pm, uint8_t* map_pr, void* stream);
/* seam fill: every texel takes the uint8 value of a covered texel at the exact minimal Euclidean distance (Meijster
 * EDT, integer arithmetic, deterministic ties) and is written as k/255 fp32: kd_out [T*T,3], pm_out / pr_out [T*T].
 * src [T*T] receives the source texel (r*T+c; itself where covered); scratch: 4*T*T int32. */
int dm_seam_fill(const uint8_t* mask, int T, const uint8_t* map_kd, const uint8_t* map_pm, const uint8_t* map_pr,
                 int32_t* scratch, int32_t* src, float* kd_out, float* pm_out, float* pr_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif
