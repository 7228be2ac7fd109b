/*
 * nerfactor_b200 -- C ABI of the B200-native NeRFactor render-and-relight hot path.
 *
 * The reference (google/nerfactor) is pure Python/TensorFlow: it has no FFI.  The
 * drop-in seam is its Python class/function surface (SURVEY.md 8b); each entry
 * point below is what a binding for one reference function would call, and cites
 * the reference code it replaces (paths relative to the reference root).
 *
 * Conventions (SURVEY.md 8b "Ownership / Errors / Threading"):
 *   - every pointer named *_d is DEVICE memory owned by the caller (contiguous,
 *     row-major, fp32 unless noted); the library never allocates or frees device
 *     memory; packed weights live in a caller-provided device buffer
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *     nothing synchronises the device
 *   - every export returns 0 on success or a negative NF_ERR_* code;
 *     nf_last_error_string(ctx) describes the last failure; no C++ exception
 *     crosses the boundary
 *   - thread-compatible per nf_ctx; one process per GPU
 */
#ifndef NERFACTOR_B200_H_
#define NERFACTOR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NF_OK 0
#define NF_ERR_INVALID_ARG (-1)
#define NF_ERR_UNSUPPORTED (-2)
#define NF_ERR_CUDA (-3)
#define NF_ERR_NO_DEVICE (-4)

/* activations of a Dense layer (nerfactor/networks/mlp.py:31-35) */
#define NF_ACT_NONE 0
#define NF_ACT_RELU 1
#define NF_ACT_SIGMOID 2
#define NF_ACT_SOFTPLUS 3

/* what a row of the MLP input is built from (fused prologue) */
#define NF_MLP_POINT 0 /* embed(xyz)                       normal/albedo/brdf_z nets */
#define NF_MLP_LVIS 1  /* embed(xyz) ++ embed(surf2l)      light-visibility net      */
#define NF_MLP_BRDF 2  /* z ++ embed(rusink(l, v))         frozen learned-BRDF net   */
#define NF_MLP_SIGMA 3 /* embed(o + t d)                   NeRF sigma net            */

/* arithmetic of the Dense contractions */
#define NF_PREC_FP32 0 /* CUDA-core FFMA, fp32 throughout (parity / small nets)   */
#define NF_PREC_F16 1  /* tcgen05 kind::f16, fp16 operands, fp32 accumulate in TMEM */
#define NF_PREC_BF16 2 /* tcgen05 kind::f16, bf16 operands, fp32 accumulate in TMEM */
#define NF_PREC_F16X3 3 /* tcgen05, fp16 hi/lo split of both operands, 3 MMA chains: ~fp32 */
#define NF_PREC_F16E 4 /* nf_sigma_fwd only: NF_PREC_F16 with the positional encoding kept as an
                          fp16 hi + lo pair (two K = 64 MMA blocks more per sample, +6.7 % tensor
                          work); weights and hidden activations are plain fp16                  */

typedef struct nf_ctx nf_ctx;
typedef struct nf_mlp nf_mlp;

/* ---- context / errors ---------------------------------------------------- */
int nf_version(void);
/* device < 0: use the current device. Fails with NF_ERR_NO_DEVICE when no
 * sm_100 GPU is present (the product path never falls back to the CPU). */
int nf_ctx_create(nf_ctx** out, int device);
int nf_ctx_destroy(nf_ctx* ctx);
const char* nf_last_error_string(const nf_ctx* ctx);
int nf_ctx_sm_count(const nf_ctx* ctx);

/* ---- networks -------------------------------------------------------------
 * nf_mlp mirrors one `mlp.Network(widths, act, skip_at)` trunk plus its output
 * `mlp.Network([out_dim], act=[out_act])` head (nerfactor/networks/mlp.py:24-50;
 * built at nerfactor/models/shape.py:79-94, nerfactor.py:128-167, brdf.py:57-66,
 * nerf.py:53-71).  Host weights are Keras-layout fp32: W[l] is [in_l, out_l]
 * row-major, b[l] is [out_l]; l = 0..depth-1 are the trunk layers (ReLU), l = depth
 * is the head.  The layer after `skip_at` takes concat(hidden, input) (mlp.py:46-49).
 */
typedef struct nf_mlp_desc {
  int kind;      /* NF_MLP_*                                                    */
  int in_dim;    /* width of the embedded input (63 / 90 / 18)                  */
  int width;     /* hidden width (128 or 256)                                   */
  int depth;     /* trunk layers (4 or 8)                                       */
  int skip_at;   /* index of the layer whose output is concatenated with input  */
  int out_dim;   /* head outputs (1..4)                                         */
  int out_act;   /* NF_ACT_* of the head                                        */
  int n_freqs_a; /* positional-encoding octaves of the first input (xyz/rusink) */
  int n_freqs_b; /* octaves of the second input (light direction), LVIS only    */
  int z_dim;     /* latent width prepended to the input, BRDF only              */
  const float* const* W; /* depth + 1 host pointers                             */
  const float* const* b; /* depth + 1 host pointers                             */
} nf_mlp_desc;

/* Packs the weights on the host (fp32 Keras layout for the FFMA kernels + the
 * swizzle-free K-major fp16/bf16 images and fp32 per-ray blocks the tcgen05
 * kernels read).  The handle owns only host memory. */
int nf_mlp_create(nf_ctx* ctx, const nf_mlp_desc* desc, nf_mlp** out);
int nf_mlp_destroy(nf_mlp* mlp);
/* Bytes of device memory the caller must provide for the packed weights. */
size_t nf_mlp_device_bytes(const nf_mlp* mlp);
/* cudaMemcpyAsync of the packed image into caller memory (256-byte aligned);
 * the handle remembers `dst_d` for the forward calls. */
int nf_mlp_upload(nf_ctx* ctx, nf_mlp* mlp, void* dst_d, void* stream);

/* ---- Stage B: per-point networks -------------------------------------------
 * out[n, out_dim] = head(trunk(embed(xyz_scale * xyz)))
 * replaces Model._pred_normal_at  nerfactor/models/shape.py:196-211 (caller adds eps)
 *          Model._pred_albedo_at  nerfactor/models/nerfactor.py:377-396 (caller: affine)
 *          Model._pred_brdf_at    nerfactor/models/nerfactor.py:398-411
 *          (and chunk_apply shape.py:184-194, Embedder embedder.py:46-47)          */
int nf_point_mlp_fwd(nf_ctx* ctx, const nf_mlp* mlp, const float* xyz_d, int n,
                     float xyz_scale, float* out_d, int precision, void* stream);

/* lvis[n, L] = sigmoid(head(trunk(embed(xyz_scale*xyz) ++ embed(l2n(lxyz - xyz)))))
 * replaces Model._calc_ldir  nerfactor/models/shape.py:128-135 (never materialised)
 *          Model._pred_lvis_at nerfactor/models/shape.py:213-237                  */
int nf_lvis_fwd(nf_ctx* ctx, const nf_mlp* mlp, const float* xyz_d, int n,
                float xyz_scale, const float* lxyz_d, int n_lights, float* lvis_d,
                int precision, void* stream);
/* Same network, but the light directions are taken from xyz_dir[n,3] while the position encoding
 * uses xyz[n,3]: the smoothness-loss evaluation of nerfactor/models/shape.py:170 /
 * nerfactor.py:225, where the reference evaluates the network at the JITTERED point with the
 * directions surf2l of the un-jittered one.  tcgen05 only (NF_PREC_F16 / NF_PREC_BF16).        */
int nf_lvis_dirs_fwd(nf_ctx* ctx, const nf_mlp* mlp, const float* xyz_d, const float* xyz_dir_d,
                     int n, float xyz_scale, const float* lxyz_d, int n_lights, float* lvis_d,
                     int precision, void* stream);

/* spec[n, L] = front_lit ? softplus(head(trunk(z ++ embed(rusink)))) : 0
 * with rusink = dir2rusink(R l2n(lxyz - xyz), R l2n(cam - xyz)), R = world2local(normal)
 * replaces Model._eval_brdf_at nerfactor/models/nerfactor.py:413-457 (up to `spec`),
 *          gen_world2local nerfactor/util/geom.py:119-149, dir2rusink geom.py:152-192 */
int nf_brdf_learned_fwd(nf_ctx* ctx, const nf_mlp* mlp, const float* xyz_d,
                        const float* normal_d, const float* cam_d, const float* z_d,
                        int n, const float* lxyz_d, int n_lights, float* spec_d,
                        int precision, void* stream);

/* ---- Stage B: rendering equation -------------------------------------------
 * rgb[n, E, 3] = tonemap(sum_l brdf[n,l,:] * lvis[n,l]*[cos>0] * light[e, idx(l), :]
 *                        * cos[n,l] * area[l])
 * replaces Model._render / integrate  nerfactor/models/nerfactor.py:315-365 and the
 * BRDF evaluation that feeds it:
 *   brdf_kind 0: Microfacet.__call__  brdf/microfacet/microfacet.py:30-111
 *                (rough_d [n,1], f0)   via nerfactor_microfacet.py:116-124
 *   brdf_kind 1: albedo/pi + spec*scale  nerfactor/models/nerfactor.py:457-461
 *                (spec_d [n,L] from nf_brdf_learned_fwd)
 * `normal_d` is the raw network output + eps; it is safe-l2-normalised inside
 * (nerfactor.py:212).  light_idx_d (may be NULL = identity) maps a light direction
 * to an env-map pixel.  tonemap = clip[0,1] then optional linear2srgb
 * (nerfactor/util/img.py:140-163).                                              */
typedef struct nf_integrate_args {
  int n, n_lights, n_envmaps, envmap_pixels;
  int brdf_kind;          /* 0 microfacet, 1 learned (spec) */
  int linear2srgb;        /* nerfactor.ini:76 */
  float f0;               /* fresnel_f0 (microfacet) */
  float spec_scale;       /* learned_brdf_scale */
  const float* xyz_d;     /* [n,3] */
  const float* normal_d;  /* [n,3] */
  const float* cam_d;     /* [n,3] ray origins = camera location */
  const float* albedo_d;  /* [n,3] */
  const float* rough_d;   /* [n,1]  (kind 0) */
  const float* spec_d;    /* [n,L]  (kind 1) */
  const float* lvis_d;    /* [n,L] */
  const float* lxyz_d;    /* [L,3] */
  const float* lareas_d;  /* [L] */
  const float* light_d;   /* [E, envmap_pixels, 3] (already clipped >= 0) */
  const int32_t* light_idx_d; /* [L] or NULL */
  float* rgb_d;           /* [n, E, 3] */
} nf_integrate_args;
int nf_integrate_fwd(nf_ctx* ctx, const nf_integrate_args* args, void* stream);

/* Backward of nf_integrate_fwd for one env-map: given d_rgb = dE/d rgb, the gradients torch
 * autograd (or TF's tape) takes through the reference formulas -- Microfacet.__call__
 * (brdf/microfacet/microfacet.py:30-111) or albedo/pi + spec*scale (nerfactor.py:457-461), then
 * nerfactor.py:315-342 -- with these conventions: the gates cos > 0, chi_d, chi_g have zero
 * derivative; divide_no_nan gives 0 value and gradient where its denominator is 0; d|x| = sign(x)
 * with sign(0) = 0; the clip to [0, 1] passes the gradient on the closed interval; linear2srgb
 * takes the slope of the selected branch; rough enters through alpha = rough^2.
 *   d_normal_d is with respect to the RAW normal_d, through both normalisations (nerfactor.py:212
 *   and microfacet.py:47); d_spec_d (brdf_kind 1) is with respect to spec_d before spec_scale;
 *   d_light_d [L,3] is summed over the n points.  No gradient is taken with respect to xyz_d,
 *   cam_d, lxyz_d or lareas_d.
 * Restrictions: n_envmaps == 1, light_idx_d == NULL, envmap_pixels == n_lights (gather the texels
 * per light first); anything else is NF_ERR_UNSUPPORTED.  `args->rgb_d` is not read: the linear
 * sum is recomputed from the inputs, nothing of the forward call needs to be kept.
 * A NULL output is neither computed nor written (d_lvis_d / d_spec_d are the [n, L] writes);
 * outputs are overwritten, not accumulated into.  workspace_d: nf_integrate_bwd_workspace_bytes()
 * bytes, needed only when d_light_d is requested (per-block partial sums of d_light, added in a
 * fixed order: results are bit-identical from run to run).  No allocation, no synchronisation
 * (CUDA-graph capturable).  The workspace query is host-only and returns 0 for an unsupported
 * argument block.                                                                              */
typedef struct nf_integrate_grads {
  const float* d_rgb_d;   /* [n,3]  upstream gradient of the tonemapped rgb                       */
  float* d_lvis_d;        /* [n,L]  or NULL                                                       */
  float* d_normal_d;      /* [n,3]  w.r.t. the raw normal_d, or NULL                              */
  float* d_albedo_d;      /* [n,3]  or NULL                                                       */
  float* d_rough_d;       /* [n]    brdf_kind 0, or NULL                                          */
  float* d_spec_d;        /* [n,L]  brdf_kind 1 (w.r.t. spec_d before spec_scale), or NULL        */
  float* d_light_d;       /* [L,3]  summed over the n points, or NULL                             */
} nf_integrate_grads;
size_t nf_integrate_bwd_workspace_bytes(const nf_integrate_args* args);
int nf_integrate_bwd(nf_ctx* ctx, const nf_integrate_args* args, const nf_integrate_grads* grads,
                     void* workspace_d, size_t workspace_bytes, void* stream);

/* One-light-at-a-time relighting: rgb_olat[n, L, 3] for the L env-maps
 * olat_inten * onehot(l) + ambient (nerfactor/models/nerfactor.py:71-84, 348-354),
 * same argument block (light_d / n_envmaps ignored). */
int nf_integrate_olat_fwd(nf_ctx* ctx, const nf_integrate_args* args, float olat_inten,
                          float ambient, float* rgb_olat_d, void* stream);

/* Fused Stage B: light-visibility network -> BRDF -> rendering equation in one call, without the
 * [n, L] light-visibility / specular tensors resident in HBM.  Replaces, for rendering, the chain
 * _pred_lvis_at -> _eval_brdf_at -> _render of nerfactor/models/nerfactor.py:217-226, 262-266,
 * 315-342 (the per-point networks -- normal, albedo, roughness / z -- are evaluated before, by
 * nf_point_mlp_fwd).  Microfacet lobe, one env-map, L <= 512, NF_PREC_F16 / BF16: ONE kernel,
 * the integral is taken in the head epilogue of the visibility network.  Otherwise the three
 * kernels run over point chunks whose rows stay L2-resident (workspace from the caller).
 * lvis_d: optional [n, L] output (NULL: visibility values are not materialised at all in the
 * single-kernel case).  rgb_d [n, E, 3].                                                      */
typedef struct nf_stageb_args {
  int n, n_lights, n_envmaps, envmap_pixels;
  int brdf_kind;          /* 0 microfacet (rough_d), 1 learned lobe (z_d + mlp_brdf)            */
  int linear2srgb, z_dim;
  float f0, spec_scale, xyz_scale;
  const float* xyz_d;     /* [n,3] */
  const float* normal_d;  /* [n,3] predicted normals */
  const float* cam_d;     /* [n,3] */
  const float* albedo_d;  /* [n,3] */
  const float* rough_d;   /* [n]   microfacet */
  const float* z_d;       /* [n, z_dim] learned lobe */
  const float* lxyz_d;    /* [L,3] */
  const float* lareas_d;  /* [L] */
  const float* light_d;   /* [E, envmap_pixels, 3] */
  const int32_t* light_idx_d; /* [L] or NULL */
  float* lvis_d;          /* [n,L] or NULL */
  float* rgb_d;           /* [n,E,3] */
  int lvis_all_lights;    /* only read when lvis_d is NULL (visibility not an output) and the
                           * precision is NF_PREC_F16 / NF_PREC_BF16.  0 (default): the visibility
                           * network runs on the FRONT-LIT lights of every point only, the ones with
                           * cos(normal, light) > -1e-5 -- nerfactor.py:329-330 multiplies the
                           * visibility of every other light by zero, so rgb_d is unchanged; the
                           * learned BRDF is evaluated on front-lit pairs only in the reference
                           * itself (nerfactor.py:429-458).  1: evaluate it for every light.
                           * 2: front-lit lights only even with lvis_d given -- lvis_d then holds
                           * front_lit * visibility, the `lvis` of nerfactor.py:330.                 */
} nf_stageb_args;
size_t nf_stageB_fused_workspace_bytes(const nf_stageb_args* args, int precision);
int nf_stageB_fused_fwd(nf_ctx* ctx, const nf_mlp* mlp_lvis, const nf_mlp* mlp_brdf,
                        const nf_stageb_args* args, int precision, void* workspace_d,
                        size_t workspace_bytes, void* stream);

/* Microfacet.__call__ (brdf/microfacet/microfacet.py:30-72) as a standalone op for callers that
 * use the class directly: brdf[n, L, 3] = GGX specular (achromatic, view-side G, f0) + albedo/pi
 * for caller-supplied directions pts2l[n, L, 3], pts2c[n, 3] and normals (all normalised inside
 * with eps 1e-6, as the reference does).  albedo_d NULL -> ones; rough_d NULL -> default_rough.
 * (The renderer, nf_integrate_fwd, fuses the same lobe and never builds [n, L, 3].)            */
int nf_microfacet_brdf_fwd(nf_ctx* ctx, const float* pts2l_d, const float* pts2c_d,
                           const float* normal_d, const float* albedo_d, const float* rough_d,
                           int n, int n_lights, float default_rough, int lambert_only, float f0,
                           float* brdf_d, void* stream);

/* ---- Stage A: rays, sigma march, compositing --------------------------------
 * rayo/rayd[h*w, 3] (fp64 math, fp32 store, ray n = y*w + x, no half-pixel offset)
 * replaces Dataset._gen_rays nerfactor/datasets/nerf.py:172-193 (ndc=False, spp=1).
 * c2w: 16 HOST doubles (row-major 4x4).  normalize != 0 additionally applies
 * tf.linalg.l2_normalize (geometry_from_nerf.py:100) to rayd.                     */
int nf_gen_rays(nf_ctx* ctx, const double* c2w_host, double cam_angle_x, int h, int w,
                int normalize, float* rayo_d, float* rayd_d, void* stream);

/* z[n, S]: t = linspace(0,1,S); z = near(1-t) + far t (or linear in disparity);
 * optional stratified perturbation with caller-supplied uniforms u_d[n,S]
 * replaces nerf.Model.gen_z nerfactor/models/nerf.py:120-136                     */
int nf_gen_z(nf_ctx* ctx, float near, float far, int n_samples, int n_rays,
             int lin_in_disp, const float* perturb_u_d, float* z_d, void* stream);

/* sigma[n, S] = in_bbox ? relu(sigma_out(enc(embed(o + z d)))) : 0
 * replaces eval_sigma_mlp nerfactor/geometry_from_nerf.py:322-350 (+ check_bounds
 * :365-378; bbox = 6 floats x0,x1,y0,y1,z0,z1 on the HOST, or NULL)               */
int nf_sigma_fwd(nf_ctx* ctx, const nf_mlp* mlp, const float* rayo_d,
                 const float* rayd_d, const float* z_d, int n_rays, int n_samples,
                 const float* bbox_host, float* sigma_d, int precision, void* stream);

/* Same as nf_sigma_fwd plus normal[n,S,3] = -l2_normalize(d sigma / d xyz)
 * replaces the GradientTape.batch_jacobian block geometry_from_nerf.py:285-305.
 * precision: NF_PREC_FP32 (CUDA cores) or NF_PREC_F16 / NF_PREC_BF16 (tcgen05 forward +
 * backward, fp32 accumulation; NF_ERR_UNSUPPORTED unless the net is 8 x 256, skip 4, F=10) */
int nf_sigma_normal_fwd(nf_ctx* ctx, const nf_mlp* mlp, const float* rayo_d,
                        const float* rayd_d, const float* z_d, int n_rays,
                        int n_samples, const float* bbox_host, float* sigma_d,
                        float* normal_d, int precision, void* stream);

/* ---- full NeRF network with viewing directions (the step before Stage A) ----
 * Colour branch of nerfactor/models/nerf.py:53-71 on top of an NF_MLP_SIGMA network:
 * bottleneck Dense(256, linear), rgb_out = Dense(128, relu) -> Dense(3, linear) on
 * concat(bottleneck, embed(view)) (Keras layouts [in, out]; n_freqs_view = 4 => 27 columns). */
typedef struct nf_nerf_rgb_desc {
  int n_freqs_view;            /* nerf.ini n_freqs_view                          */
  int hidden;                  /* mlp_width // 2                                 */
  const float* w_bottleneck;   /* [256, 256]                                     */
  const float* b_bottleneck;   /* [256]                                          */
  const float* w_rgb0;         /* [256 + 3 (1 + 2 n_freqs_view), hidden]         */
  const float* b_rgb0;         /* [hidden]                                       */
  const float* w_rgb1;         /* [hidden, 3]                                    */
  const float* b_rgb1;         /* [3]                                            */
} nf_nerf_rgb_desc;
/* Appends the colour-branch operand images to a packed sigma network; call between
 * nf_mlp_create and nf_mlp_device_bytes / nf_mlp_upload.                                  */
int nf_mlp_attach_rgb(nf_ctx* ctx, nf_mlp* sigma_mlp, const nf_nerf_rgb_desc* rgb);
/* rgbs[n, S, 4] = (raw r, g, b, raw sigma) at the samples o + z d, views = d:
 * replaces Model._eval_nerf_at nerfactor/models/nerf.py:254-290 (use_views = True); the
 * caller composites with nf_composite (sigmoid / ReLU applied there, nerf.py:214-252).
 * tcgen05 only (NF_PREC_F16 / NF_PREC_BF16).                                              */
int nf_nerf_fwd(nf_ctx* ctx, const nf_mlp* mlp, const float* rayo_d, const float* rayd_d,
                const float* z_d, int n_rays, int n_samples, float* rgbs_d, int precision,
                void* stream);

/* weights[n,S] (optional), occu[n], depth[n], surf[n,3] (optional),
 * exp_normal[n,3] (optional, needs normal_d [n,S,3])
 * replaces nerf.Model.accumulate_sigma nerfactor/models/nerf.py:184-212 (noise 0) and
 * the reductions geometry_from_nerf.py:312-317, :134                              */
int nf_composite(nf_ctx* ctx, const float* sigma_d, const float* z_d,
                 const float* rayo_d, const float* rayd_d, const float* normal_d,
                 int n_rays, int n_samples, float* weights_d, float* occu_d,
                 float* depth_d, float* surf_d, float* exp_normal_d, void* stream);

/* z_all[n, S_c + S_f] = sort(concat(z_c, inv_transform_sample(mid(z_c), w[1:-1])))
 * replaces nerf.Model.gen_z_fine nerfactor/models/nerf.py:138-147 and
 * inv_transform_sample nerfactor/util/math.py:71-94 (det=True)                    */
int nf_gen_z_fine(nf_ctx* ctx, const float* z_coarse_d, const float* weights_d,
                  int n_rays, int n_coarse, int n_fine, float* z_all_d, void* stream);

/* Light-visibility march set-up: for every (point, light) pair writes the ray
 * origin/direction (surf, l2_normalize(lxyz - surf)) and front-lit flag
 * ((surf2l . normal) > 0), replaces geometry_from_nerf.py:196-215.                */
int nf_lvis_rays(nf_ctx* ctx, const float* surf_d, const float* normal_d, int n_pts,
                 const float* lxyz_d, int n_lights, float* rayo_d, float* rayd_d,
                 uint8_t* front_lit_d, void* stream);

/* ---- whole ray marches in one call (intermediates in a caller-provided workspace) ----------
 * Camera -> surface: gen_z -> sigma (coarse net) -> weights -> inverse-CDF resampling -> sigma and
 * d sigma / dx normals (fine net) on the sorted union -> occu[n], depth[n], normal[n, 3]
 * (= sum w, sum w z, sum w n).  Replaces compute_depth_and_normal
 * nerfactor/geometry_from_nerf.py:249-319; n_coarse / n_fine are the ACTUAL counts (the reference
 * adds 64 to the .ini values, :250-251).  precision as nf_sigma_fwd (NF_PREC_F16E applies to the
 * coarse pass; the gradient kernel then runs NF_PREC_F16).  Rays are processed in chunks; the
 * workspace holds one chunk's [c, S] buffers.                                                   */
size_t nf_raymarch_depth_normal_workspace_bytes(int n_rays, int n_coarse, int n_fine);
int nf_raymarch_depth_normal_fwd(nf_ctx* ctx, const nf_mlp* mlp_coarse, const nf_mlp* mlp_fine,
                                 const float* rayo_d, const float* rayd_d, int n_rays, float near,
                                 float far, int n_coarse, int n_fine, int lin_in_disp,
                                 const float* bbox_host, int precision, void* workspace_d,
                                 size_t workspace_bytes, float* occu_d, float* depth_d,
                                 float* normal_d, void* stream);
/* Surface -> light: lvis[n_pts, L] = 1 - sum w of the hierarchical march from surf towards every
 * light with (surf2l . normal) > 0, 0 for back-lit pairs.  Front-lit test, compaction, both
 * marches and the scatter run on the device.  Replaces compute_light_visibility
 * nerfactor/geometry_from_nerf.py:177-246 (all lights at once instead of its per-light loop).
 * NOTE: synchronises `stream` once per chunk of 2^19 pairs to read the number of front-lit pairs
 * (it sizes the march launches) -- the one op of this library that does.                        */
size_t nf_raymarch_lvis_workspace_bytes(int n_pts, int n_lights, int n_coarse, int n_fine);
int nf_raymarch_lvis_fwd(nf_ctx* ctx, const nf_mlp* mlp_coarse, const nf_mlp* mlp_fine,
                         const float* surf_d, const float* normal_d, int n_pts,
                         const float* lxyz_d, int n_lights, float lvis_near, float lvis_far,
                         int n_coarse, int n_fine, int lin_in_disp, const float* bbox_host,
                         int precision, void* workspace_d, size_t workspace_bytes, float* lvis_d,
                         void* stream);

/* Input rows of the light-visibility network for the train step, materialised in one launch
 * (the training path runs the network layer by layer on materialised activations):
 *   out[(i, l), :] = [embed(xyz_scale xyz_i) | embed(l2n(lxyz_l - xyz_dir_i)) | 0 ...]  (row stride ld)
 * replaces _calc_ldir + the two Embedder calls + tf.concat of shape.py:128-135, 213-233;
 * xyz_dir = xyz for the clean evaluation, the un-jittered point for the jittered one (:170).   */
int nf_lvis_inputs_fwd(nf_ctx* ctx, const float* xyz_d, const float* xyz_dir_d, int n,
                       const float* lxyz_d, int n_lights, float xyz_scale, int n_freqs_xyz,
                       int n_freqs_ldir, int ld, float* out_d, void* stream);

/* ---- training (config 4): Dense layers on materialised activations + optimizer ----
 * One Keras Dense of mlp.Network (nerfactor/networks/mlp.py:34, 39-50) at a time:
 *   y[m, n] = act([x1[m,k1] | x2[m,k2]] w[(k1+k2), n] + b[n])      (x2 = skip concat, k2 may be 0)
 * n, k1, k2 must be multiples of 4 (pad heads / embeddings with zero rows / columns).
 * precision: NF_PREC_FP32 (CUDA cores) or NF_PREC_F16 / NF_PREC_BF16 (tcgen05: operands rounded
 * to 16 bit, fp32 accumulation, fp32 inputs / outputs; shapes the tensor-core kernels do not
 * cover -- more than 256 input or output features -- silently use the FP32 kernels).
 * work_d: caller scratch of nf_dense_fwd_workspace_bytes() bytes (may be NULL when that is 0). */
size_t nf_dense_fwd_workspace_bytes(int n, int k1, int k2, int precision);
int nf_dense_fwd(nf_ctx* ctx, const float* x1_d, int k1, const float* x2_d, int k2,
                 const float* w_d, const float* b_d, long long m, int n, int act, float* y_d,
                 void* work_d, int precision, void* stream);
/* Backward of nf_dense_fwd (what tape.gradient computes for one Dense,
 * nerfactor/trainvali.py:278-285): with dz = dy * act'(y),
 *   dx1 | dx2 = dz w^T (either may be NULL), dw += [x1 | x2]^T dz, db += colsum(dz)
 * (dw_d / db_d are ACCUMULATED into and may be NULL).  work_d: caller scratch of
 * nf_dense_bwd_workspace_bytes(m, n, k1, k2, precision) bytes.                         */
size_t nf_dense_bwd_workspace_bytes(long long m, int n, int k1, int k2, int precision);
int nf_dense_bwd(nf_ctx* ctx, const float* x1_d, int k1, const float* x2_d, int k2,
                 const float* w_d, const float* y_d, const float* dy_d, long long m, int n,
                 int act, float* dx1_d, float* dx2_d, float* dw_d, float* db_d, void* work_d,
                 int precision, void* stream);
/* ---- whole-network forward / backward of the train step (the `*_bwd` counterparts of the
 * per-network forward ops; SURVEY 8b).  One call runs every Dense of an mlp.Network
 * (nerfactor/networks/mlp.py:39-50: `depth - 1` hidden layers, the input re-concatenated as
 * [h | x] in front of layer `skip_layer`, + the seq.Network head) and what tape.gradient
 * (nerfactor/trainvali.py:278-285) computes for it.  Activations stay 16-bit rows inside
 * `workspace_d` (nf_mlp_chain_workspace_bytes; the SAME workspace must be passed to the backward
 * call, untouched in between).  x_d [rows, in_dim] (in_dim % 4 == 0: pad with zero columns and zero
 * weight rows), y_d [rows, width[depth-1]] (head width % 4 == 0: pad W / b with zero columns);
 * hidden widths % 16 == 0, every layer input <= 256 columns; NF_PREC_F16 / NF_PREC_BF16 only.
 * Backward: dy_d like y_d; dx_d [rows, in_dim] or NULL; dw_d[l] / db_d[l] (Keras layout; the
 * skip layer's W is [width[skip-1] + in_dim, width[skip]]) are ACCUMULATED INTO (+=), NULL
 * entries / NULL arrays are skipped.  Replaces the per-layer nf_dense_fwd / nf_dense_bwd sequence
 * for networks of this shape; numbers agree with it up to the rounding of the bias-gradient sums. */
#define NF_CHAIN_MAX 8
typedef struct nf_mlp_chain {
  int depth;                     /* Dense layers incl. the head, 2..NF_CHAIN_MAX */
  int in_dim;
  int skip_layer;                /* index of the layer fed with [h | x]; 0 = no skip */
  int width[NF_CHAIN_MAX];
  int act[NF_CHAIN_MAX];         /* NF_ACT_* */
  const float* w[NF_CHAIN_MAX];  /* device, fp32 */
  const float* b[NF_CHAIN_MAX];
} nf_mlp_chain;
size_t nf_mlp_chain_workspace_bytes(const nf_mlp_chain* chain, long long rows);
int nf_mlp_chain_fwd(nf_ctx* ctx, const nf_mlp_chain* chain, const float* x_d, long long rows,
                     float* y_d, void* workspace_d, int precision, void* stream);
int nf_mlp_chain_bwd(nf_ctx* ctx, const nf_mlp_chain* chain, long long rows, const float* y_d,
                     const float* dy_d, float* dx_d, float* const* dw_d, float* const* db_d,
                     void* workspace_d, int precision, void* stream);

/* One AMSGrad-Adam update of a flat parameter buffer: tf.keras.optimizers.Adam(lr, amsgrad=True)
 * as configured at nerfactor/trainvali.py:110-127 (beta1 .9, beta2 .999, epsilon 1e-7);
 * `step` is the 1-based iteration count, `lr` the already-decayed learning rate.          */
int nf_adam_amsgrad_step(nf_ctx* ctx, float* param_d, const float* grad_d, float* m_d, float* v_d,
                         float* vhat_d, long long count, float lr, float beta1, float beta2,
                         float eps, long long step, void* stream);

/* ---- diagnostics (no reference counterpart) ---------------------------------
 * One 128x128xK tcgen05 tile: out[128,128] = a[128,K] * b[128,K]^T through the same
 * TMEM / shared-memory operand layouts the fused kernels use (bring-up check).   */
int nf_selftest_umma(nf_ctx* ctx, const float* a_d, const float* b_d, int K,
                     int swap_lbo_sbo, float* out_d, void* stream);
/* Same through one CTA-pair MMA (cta_group::2): out[256,128] = a[256,K] * b[128,K]^T.   */
int nf_selftest_umma2(nf_ctx* ctx, const float* a_d, const float* b_d, int K, float* out_d,
                      void* stream);

/* TMEM read / write throughput on one SM (tcgen05.ld / .st), alone or under a concurrent
 * tcgen05.mma stream: out_d[0] = reader cycles, out_d[1] = MMA-stream cycles (device int64[4]).
 * mode bits: 1 loads, 2 stores, 4 MMA stream, 8 loads as .x16, 16 MMA N = 256.               */
int nf_selftest_tmem(nf_ctx* ctx, int reader_warps, int iters, int mma_iters, int mode,
                     long long* out_d, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NERFACTOR_B200_H_ */
