// Backward of the rendering equation (nf_integrate_fwd with one env-map): the gradients torch
// autograd / TF's tape take through
//   Model._render / integrate    nerfactor/models/nerfactor.py:315-342 (front-lit gate, the
//                                hemisphere sum, clip, linear2srgb),
//   Microfacet.__call__          brdf/microfacet/microfacet.py:30-111 (brdf_kind 0), or
//   albedo / pi + spec * scale   nerfactor/models/nerfactor.py:457-461 (brdf_kind 1),
//   and the normalisation of the raw normal (nerfactor.py:212).
//
// Layout as in the forward kernel (nf_integrate.cu): a warp owns one point at a time and its lanes
// stride the lights; light positions, areas and texels sit in shared memory.  Two passes over the
// point's lvis / spec row: the first re-forms the linear sum and hence the upstream gradient g of
// the un-tonemapped colour; the second, over the same row while it is still in L1 / L2, writes the
// per-pair gradients and accumulates the per-point sums, which end in warp shuffle reductions.
// d_light is a reduction over points: every warp keeps its partial sums in its own slice of shared
// memory (a lane owns the lights lane, lane + 32, ...), the block sums its warps in order into the
// caller's workspace, and a second kernel sums the blocks in order -- no float atomics, so results
// are bit-identical from run to run.
//
// Scalar fp32 on the reference formulas.  The one rewrite is the GGX distribution term, formed as
//   D = a2 chi / (pi u^2),  u = a2 cm^2 + |h x n|^2    (pi u^2 = pi cm^4 (a2 + tan^2)^2 for cm != 0),
// and differentiated in that form; both have the same value and derivatives wherever the
// reference's denominator is non-zero (where it is zero, divide_no_nan gives value and gradient 0,
// and so does this kernel).
#include <algorithm>

#include "nf_common.cuh"

namespace {

constexpr int BWD_MAX_BLOCKS = 1024;   // cap of the grid, and of the d_light partials it writes

// warps per block: the largest count whose d_light slices still fit next to the light arrays
// (7 L + 3 L warps floats) in 227 KB of shared memory at the op's n_lights cap of 4096
__host__ __device__ inline int bwd_warps(int n_lights) {
  return n_lights <= 1024 ? 8 : (n_lights <= 2048 ? 4 : 2);
}

// upper bound of the grid, and of the d_light partials in the workspace: one block per `warps`
// points, at most BWD_MAX_BLOCKS (host-only; the launch may use fewer blocks)
inline int bwd_max_blocks(int n, int n_lights) {
  const int w = bwd_warps(n_lights);
  return (int)std::min<long long>(((long long)n + w - 1) / w, BWD_MAX_BLOCKS);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;   // butterfly: every lane ends with the same bits
}

__device__ __forceinline__ float sgnf(float x) { return x > 0.f ? 1.f : (x < 0.f ? -1.f : 0.f); }

// adjoint of y = x * rsqrt(max(|x|^2, eps)) (tf.linalg.l2_normalize, util/math.py:63-64)
__device__ __forceinline__ f3 l2n_bwd(f3 x, f3 dy, float eps) {
  const float sq = dot3(x, x);
  const float s = 1.0f / sqrtf(fmaxf(sq, eps));
  const float k = sq >= eps ? s * s * s * dot3(x, dy) : 0.f;
  return mk3(dy.x * s - k * x.x, dy.y * s - k * x.y, dy.z * s - k * x.z);
}

// d tonemap(x) / dx: clip to [0, 1] (gradient on the closed interval, as tf.clip_by_value and
// torch.clamp), then the slope of the sRGB branch that is selected (nerfactor/util/img.py:140-163)
__device__ __forceinline__ float tonemap_grad(float x, int srgb) {
  if (!(x >= 0.f && x <= 1.f)) return 0.f;
  if (!srgb) return 1.f;
  return x <= 0.0031308f ? 12.92f : (1.055f / 2.4f) * powf(x, 1.0f / 2.4f - 1.0f);
}

struct Point {             // per-point constants (every lane of the warp holds the same values)
  f3 p, nraw, n1, n2, v2, lam;
  bool n_unit;             // n2 is a unit vector (the raw normal is not ~0)
  float rough, alpha, a2;  // rough, alpha = rough^2, a2 = alpha^2          (microfacet.py:54)
  float cv, cv2_raw, cv2, tv2_raw, tv2, q, sq, dg;   // view side of G       (microfacet.py:74-91)
};

__device__ __forceinline__ Point load_point(const nf_integrate_args& a, int i) {
  Point c;
  c.p = ld3(a.xyz_d + (size_t)i * 3);
  c.nraw = ld3(a.normal_d + (size_t)i * 3);
  c.n1 = l2n(c.nraw, 1e-6f);                                     // nerfactor.py:212
  const f3 v1 = l2n(ld3(a.cam_d + (size_t)i * 3) - c.p, 1e-6f);  // shape.py:137-144
  const f3 alb = ld3(a.albedo_d + (size_t)i * 3);
  c.lam = mk3(alb.x / NF_PI_F, alb.y / NF_PI_F, alb.z / NF_PI_F);
  c.n2 = c.n1; c.v2 = v1;
  c.n_unit = dot3(c.n1, c.n1) >= 1e-6f;
  c.rough = c.alpha = c.a2 = c.cv = c.cv2_raw = c.cv2 = c.tv2_raw = c.tv2 = c.q = c.sq = c.dg = 0.f;
  if (a.brdf_kind == 0) {
    c.n2 = l2n(c.n1, 1e-6f);                                     // microfacet.py:47-49
    c.v2 = l2n(v1, 1e-6f);
    c.rough = a.rough_d[i];
    c.alpha = c.rough * c.rough;
    c.a2 = c.alpha * c.alpha;
    c.cv = dot3(c.n2, c.v2);                                     // :77
    c.cv2_raw = c.cv * c.cv;
    c.cv2 = fminf(fmaxf(c.cv2_raw, 0.f), 1.f);                   // :82-84
    c.tv2_raw = divide_no_nan(1.f - c.cv2, c.cv2);               // :85-87
    c.tv2 = fmaxf(c.tv2_raw, 0.f);
    c.q = 1.f + c.a2 * c.tv2;
    c.sq = sqrtf(c.q);
    c.dg = 1.f + c.sq;                                           // :88-89 (>= 2)
  }
  return c;
}

struct Pair {
  f3 l;              // unit direction to the light (shape.py:128-135)
  float cos, w;      // l . n1 and [cos > 0] lvis cos area (nerfactor.py:325-336)
  float spec;        // achromatic specular term of the BRDF
  // microfacet only: what the adjoint needs
  f3 l2, h;
  float f, cm, u, dn, chi_g, ldn, den;
};

template <int KIND>
__device__ __forceinline__ Pair eval_pair(const nf_integrate_args& a, const Point& c,
                                          const float* sx, const float* sy, const float* sz,
                                          const float* sa, int l, float lvis, float spec_in) {
  Pair r;
  r.l = l2n(mk3(sx[l], sy[l], sz[l]) - c.p, 1e-6f);
  r.cos = dot3(r.l, c.n1);
  r.w = (r.cos > 0.f ? lvis : 0.f) * r.cos * sa[l];
  if (KIND == 0) {
    r.l2 = l2n(r.l, 1e-6f);                                      // microfacet.py:46
    const f3 hs = r.l2 + c.v2;
    const float hh = dot3(hs, hs);
    r.h = hs * (1.0f / sqrtf(fmaxf(hh, 1e-6f)));                 // :51-52
    const float om = 1.f - dot3(r.l2, r.h);
    const float om2 = om * om;
    r.f = a.f0 + (1.f - a.f0) * (om2 * om2 * om);                // :106-111
    r.cm = dot3(r.h, c.n2);                                      // :96
    const float cm2 = r.cm * r.cm;
    // 1 - cm^2 as |h x n|^2 (h, n unit): near the lobe's peak 1 - cm^2 cancels to a rounding error
    // comparable with a2 itself at low roughness
    const f3 hxn = cross3(r.h, c.n2);
    r.u = fmaf(c.a2, cm2, (hh >= 1e-6f && c.n_unit) ? dot3(hxn, hxn) : 1.f - cm2);
    // dn = 1 / (pi u^2); D = a2 dn where chi_d = [cm > 0] and u != 0, else 0   (:93-104)
    r.dn = (r.cm > 0.f && r.u != 0.f) ? 1.f / (NF_PI_F * (r.u * r.u)) : 0.f;
    const float d = c.a2 * r.dn;
    const float hv = dot3(r.h, c.v2);                            // :78-81
    r.chi_g = (c.cv != 0.f && hv / c.cv > 0.f) ? 1.f : 0.f;
    const float g = r.chi_g * 2.f / c.dg;
    r.ldn = dot3(r.l2, c.n2);
    r.den = 4.f * fabsf(r.ldn) * fabsf(c.cv);                    // :58-61
    r.spec = r.den != 0.f ? r.f * g * d / r.den : 0.f;
  } else {
    r.spec = spec_in * a.spec_scale;                             // nerfactor.py:460
  }
  return r;
}

// smem (floats): X[L] Y[L] Z[L] AREA[L] R[L] G[L] B[L], then (d_light requested) one [3][L]
// slice per warp.  `part`: [gridDim.x][3][L] block partials of d_light, or NULL.
template <int KIND>
__global__ void __launch_bounds__(256) integrate_bwd_kernel(const nf_integrate_args a,
                                                            const nf_integrate_grads gr,
                                                            float* __restrict__ part) {
  extern __shared__ float smf[];
  const int L = a.n_lights;
  float* sx = smf; float* sy = sx + L; float* sz = sy + L; float* sa = sz + L;
  float* sr = sa + L; float* sg = sr + L; float* sb = sg + L;
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* dl = part ? sb + L + (size_t)warp * 3 * L : nullptr;     // this warp's d_light slice
  for (int l = threadIdx.x; l < L; l += blockDim.x) {
    sx[l] = a.lxyz_d[l * 3]; sy[l] = a.lxyz_d[l * 3 + 1]; sz[l] = a.lxyz_d[l * 3 + 2];
    sa[l] = a.lareas_d[l];
    sr[l] = a.light_d[l * 3]; sg[l] = a.light_d[l * 3 + 1]; sb[l] = a.light_d[l * 3 + 2];
  }
  if (part)
    for (int k = lane; k < 3 * L; k += 32) dl[k] = 0.f;
  __syncthreads();

  for (int i = blockIdx.x * nw + warp; i < a.n; i += gridDim.x * nw) {
    const Point c = load_point(a, i);
    const float* lv = a.lvis_d + (size_t)i * L;
    const float* sp = KIND == 1 ? a.spec_d + (size_t)i * L : nullptr;
    // ---- pass 1: the linear sum (nerfactor.py:334-336) and sum_l w light / pi (for d_albedo)
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, wl0 = 0.f, wl1 = 0.f, wl2 = 0.f;
    for (int l = lane; l < L; l += 32) {
      const Pair r = eval_pair<KIND>(a, c, sx, sy, sz, sa, l, __ldg(lv + l),
                                     KIND == 1 ? __ldg(sp + l) : 0.f);
      const float w0 = r.w * sr[l], w1 = r.w * sg[l], w2 = r.w * sb[l];
      s0 = fmaf(r.spec + c.lam.x, w0, s0); wl0 += w0;
      s1 = fmaf(r.spec + c.lam.y, w1, s1); wl1 += w1;
      s2 = fmaf(r.spec + c.lam.z, w2, s2); wl2 += w2;
    }
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
    const f3 drgb = ld3(gr.d_rgb_d + (size_t)i * 3);
    const float g0 = drgb.x * tonemap_grad(s0, a.linear2srgb);
    const float g1 = drgb.y * tonemap_grad(s1, a.linear2srgb);
    const float g2 = drgb.z * tonemap_grad(s2, a.linear2srgb);
    const bool live = g0 != 0.f || g1 != 0.f || g2 != 0.f;     // warp-uniform

    // ---- pass 2: per-pair gradients, per-point sums
    f3 dn1 = mk3(0.f, 0.f, 0.f), dn2 = mk3(0.f, 0.f, 0.f);
    float da2 = 0.f, dcv_abs = 0.f, dgsum = 0.f;
    for (int l = lane; l < L; l += 32) {
      if (!live) {
        if (gr.d_lvis_d) gr.d_lvis_d[(size_t)i * L + l] = 0.f;
        if (KIND == 1 && gr.d_spec_d) gr.d_spec_d[(size_t)i * L + l] = 0.f;
        continue;
      }
      const float lvis = __ldg(lv + l);
      const Pair r = eval_pair<KIND>(a, c, sx, sy, sz, sa, l, lvis, KIND == 1 ? __ldg(sp + l) : 0.f);
      const float L0 = sr[l], L1 = sg[l], L2 = sb[l];
      const float b0 = r.spec + c.lam.x, b1 = r.spec + c.lam.y, b2 = r.spec + c.lam.z;
      const float gbl = g0 * b0 * L0 + g1 * b1 * L1 + g2 * b2 * L2;
      const float t = r.cos > 0.f ? gbl * sa[l] : 0.f;           // d contrib / d (lvis cos)
      if (gr.d_lvis_d) gr.d_lvis_d[(size_t)i * L + l] = t * r.cos;
      if (dl) {
        dl[l] += g0 * b0 * r.w;
        dl[L + l] += g1 * b1 * r.w;
        dl[2 * L + l] += g2 * b2 * r.w;
      }
      const float dcos = t * lvis;                                 // nerfactor.py:325
      dn1 = dn1 + r.l * dcos;
      const float dspec = r.w * (g0 * L0 + g1 * L1 + g2 * L2);     // d rgb / d spec (pre-tonemap)
      if (KIND == 1) {
        if (gr.d_spec_d) gr.d_spec_d[(size_t)i * L + l] = a.spec_scale * dspec;
      } else if (r.den != 0.f) {
        // spec = divide_no_nan(F G D, 4 |l.n| |v.n|)                  microfacet.py:58-61
        const float rr = dspec / r.den;
        const float d = c.a2 * r.dn;
        const float g = r.chi_g * 2.f / c.dg;
        const float dd = rr * r.f * g;                             // d spec / d D
        dgsum += rr * r.f * d * r.chi_g;                           // d spec / d G, times chi_g
        const float dden = -rr * r.spec;
        const float dldn = dden * 4.f * fabsf(c.cv) * sgnf(r.ldn);
        dcv_abs += dden * 4.f * fabsf(r.ldn);
        dn2 = dn2 + r.l2 * dldn;
        if (r.dn != 0.f) {
          // D = a2 dn, u = a2 cm^2 + 1 - cm^2:  dD/da2 = dn - 2 D cm^2 / u,
          // dD/dcm = -4 D (a2 - 1) cm / u                            (:93-104)
          const float iu = 1.f / r.u;
          da2 += dd * (r.dn - 2.f * d * (r.cm * r.cm) * iu);
          dn2 = dn2 + r.h * (dd * (-4.f * d * (c.a2 - 1.f) * r.cm * iu));
        }
      }
    }
    dn1.x = warp_sum(dn1.x); dn1.y = warp_sum(dn1.y); dn1.z = warp_sum(dn1.z);
    float drough = 0.f;
    if (KIND == 0) {
      dn2.x = warp_sum(dn2.x); dn2.y = warp_sum(dn2.y); dn2.z = warp_sum(dn2.z);
      da2 = warp_sum(da2); dcv_abs = warp_sum(dcv_abs); dgsum = warp_sum(dgsum);
      // G = divide_no_nan(2 chi_g, 1 + sqrt(1 + a2 tan^2_v)) with its per-point denominator
      const float ddg = -dgsum * 2.f / (c.dg * c.dg);
      const float dq = ddg * 0.5f / c.sq;
      da2 += dq * c.tv2;
      const float dt = c.tv2_raw >= 0.f ? dq * c.a2 : 0.f;                       // clip(min=0)
      const float dcv2 = c.cv2 != 0.f ? -dt / c.cv2 - dt * c.tv2_raw / c.cv2 : 0.f;  // divide_no_nan
      float dcv = (c.cv2_raw >= 0.f && c.cv2_raw <= 1.f) ? dcv2 * 2.f * c.cv : 0.f;  // clip [0, 1]
      dcv += dcv_abs * sgnf(c.cv);                                                // |v.n|
      dn2 = dn2 + c.v2 * dcv;
      dn1 = dn1 + l2n_bwd(c.n1, dn2, 1e-6f);                     // microfacet.py:47-49
      drough = da2 * 2.f * c.alpha * 2.f * c.rough;              // a2 = (rough^2)^2
    }
    if (gr.d_normal_d && lane == 0) {
      const f3 dn = l2n_bwd(c.nraw, dn1, 1e-6f);                 // nerfactor.py:212
      float* o = gr.d_normal_d + (size_t)i * 3;
      o[0] = dn.x; o[1] = dn.y; o[2] = dn.z;
    }
    if (gr.d_albedo_d) {
      wl0 = warp_sum(wl0); wl1 = warp_sum(wl1); wl2 = warp_sum(wl2);
      if (lane == 0) {
        float* o = gr.d_albedo_d + (size_t)i * 3;
        o[0] = g0 * wl0 / NF_PI_F; o[1] = g1 * wl1 / NF_PI_F; o[2] = g2 * wl2 / NF_PI_F;
      }
    }
    if (KIND == 0 && gr.d_rough_d && lane == 0) gr.d_rough_d[i] = drough;
  }

  if (part) {
    __syncthreads();
    float* out = part + (size_t)blockIdx.x * 3 * L;
    const float* s0 = sb + L;
    for (int k = threadIdx.x; k < 3 * L; k += blockDim.x) {
      float s = 0.f;
      for (int w = 0; w < nw; ++w) s += s0[(size_t)w * 3 * L + k];
      out[k] = s;
    }
  }
}

// d_light[l, c] = sum over blocks b, in order, of part[b][c][l]
__global__ void __launch_bounds__(256) integrate_bwd_light_reduce(const float* __restrict__ part,
                                                                  int n_blocks, int L,
                                                                  float* __restrict__ d_light) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= 3 * L) return;
  float s = 0.f;
#pragma unroll 8
  for (int b = 0; b < n_blocks; ++b) s += part[(size_t)b * 3 * L + k];
  const int c = k / L, l = k % L;
  d_light[(size_t)l * 3 + c] = s;
}

}  // namespace

extern "C" {

size_t nf_integrate_bwd_workspace_bytes(const nf_integrate_args* a) {
  if (!a || a->n <= 0 || a->n_lights <= 0 || a->n_lights > 4096 || a->n_envmaps != 1) return 0;
  return (size_t)bwd_max_blocks(a->n, a->n_lights) * 3 * (size_t)a->n_lights * sizeof(float);
}

int nf_integrate_bwd(nf_ctx* ctx, const nf_integrate_args* a, const nf_integrate_grads* g,
                     void* workspace_d, size_t workspace_bytes, void* stream) {
  NF_CHECK_ARG(ctx, a && g, "null args / grads");
  NF_CHECK_ARG(ctx, a->n >= 0 && a->n_lights > 0 && a->n_lights <= 4096, "bad n / n_lights");
  NF_CHECK_ARG(ctx, a->brdf_kind == 0 || a->brdf_kind == 1, "bad brdf_kind");
  if (a->n_envmaps != 1 || a->light_idx_d != nullptr || a->envmap_pixels != a->n_lights)
    return nf_set_error(ctx, NF_ERR_UNSUPPORTED,
                        "%s: the backward pass takes one env-map of n_lights texels "
                        "(n_envmaps == 1, light_idx_d == NULL, envmap_pixels == n_lights)", __func__);
  NF_CHECK_ARG(ctx, a->brdf_kind == 0 || !g->d_rough_d, "d_rough_d needs brdf_kind 0");
  NF_CHECK_ARG(ctx, a->brdf_kind == 1 || !g->d_spec_d, "d_spec_d needs brdf_kind 1");
  cudaStream_t st = (cudaStream_t)stream;
  const int L = a->n_lights;
  if (a->n == 0) {
    if (g->d_light_d) NF_CUDA(ctx, cudaMemsetAsync(g->d_light_d, 0, sizeof(float) * 3 * L, st));
    return NF_OK;
  }
  NF_CHECK_ARG(ctx, a->xyz_d && a->normal_d && a->cam_d && a->albedo_d && a->lvis_d && a->lxyz_d &&
                        a->lareas_d && a->light_d && g->d_rgb_d, "null buffer");
  NF_CHECK_ARG(ctx, a->brdf_kind == 0 ? a->rough_d != nullptr : a->spec_d != nullptr,
               "missing rough_d / spec_d");
  const int max_blocks = bwd_max_blocks(a->n, L);
  if (g->d_light_d) {
    const size_t need = (size_t)max_blocks * 3 * L * sizeof(float);
    NF_CHECK_ARG(ctx, workspace_d && workspace_bytes >= need,
                 "workspace smaller than nf_integrate_bwd_workspace_bytes()");
  }
  const int warps = bwd_warps(L);
  const size_t sm = sizeof(float) * (size_t)L * (7 + (g->d_light_d ? 3 * warps : 0));
  NF_CHECK_ARG(ctx, sm <= ctx->smem_optin, "n_lights too large for shared memory");
  float* part = g->d_light_d ? (float*)workspace_d : nullptr;
  int grid = 0;
#define NF_LAUNCH_BWD(KIND)                                                                        \
  do {                                                                                             \
    NF_CUDA(ctx, cudaFuncSetAttribute(integrate_bwd_kernel<KIND>,                                  \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));     \
    int per_sm = 1;                                                                                \
    NF_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(                                    \
                     &per_sm, integrate_bwd_kernel<KIND>, warps * 32, sm));                        \
    grid = ctx->sm_count * (per_sm > 0 ? per_sm : 1);                                              \
    if (grid > max_blocks) grid = max_blocks;                                                      \
    integrate_bwd_kernel<KIND><<<grid, warps * 32, sm, st>>>(*a, *g, part);                        \
  } while (0)
  if (a->brdf_kind == 0) NF_LAUNCH_BWD(0);
  else NF_LAUNCH_BWD(1);
#undef NF_LAUNCH_BWD
  NF_LAUNCH_CHECK(ctx);
  if (g->d_light_d) {
    integrate_bwd_light_reduce<<<(3 * L + 255) / 256, 256, 0, st>>>(part, grid, L, g->d_light_d);
    NF_LAUNCH_CHECK(ctx);
  }
  return NF_OK;
}

}  // extern "C"
