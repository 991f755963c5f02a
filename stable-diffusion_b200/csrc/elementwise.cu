// Streaming layout / elementwise kernels around the tensor-core ops (all HBM/L2-bound, grid-stride,
// grids sized in multiples of the SM count).
#include "../../include/sdb200.h"
#include "host.h"
#include <cuda_fp16.h>

namespace sdb {

static inline int grid_for(size_t n, int threads = 256) {
  size_t b = (n + threads - 1) / threads;
  size_t cap = static_cast<size_t>(sm_count()) * 16;
  return static_cast<int>(b < 1 ? 1 : (b > cap ? cap : b));
}
#define GRID_STRIDE(i, n)                                                                      \
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < (n); \
       i += static_cast<size_t>(gridDim.x) * blockDim.x)

// NCHW -> NHWC through a 32x32 smem tile (coalesced both ways). grid = (hw/32, c/32, nb)
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ x, int c, int hw, float* __restrict__ o32,
                                    __half* __restrict__ o16) {
  __shared__ float tile[32][33];
  int n = blockIdx.z;
  int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int cc = c0 + j, p = p0 + threadIdx.x;
    tile[j][threadIdx.x] = (cc < c && p < hw) ? x[(static_cast<size_t>(n) * c + cc) * hw + p] : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int p = p0 + j, cc = c0 + threadIdx.x;
    if (p < hw && cc < c) {
      float v = tile[threadIdx.x][j];
      size_t o = (static_cast<size_t>(n) * hw + p) * c + cc;
      if (o32) o32[o] = v;
      if (o16) o16[o] = __float2half_rn(v);
    }
  }
}
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ x, int c, int hw, float* __restrict__ out) {
  __shared__ float tile[32][33];
  int n = blockIdx.z;
  int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int p = p0 + j, cc = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (cc < c && p < hw) ? x[(static_cast<size_t>(n) * hw + p) * c + cc] : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int cc = c0 + j, p = p0 + threadIdx.x;
    if (p < hw && cc < c) out[(static_cast<size_t>(n) * c + cc) * hw + p] = tile[threadIdx.x][j];
  }
}

// 3x3 conv patches, stride 1, zero pad 1: NHWC fp32 -> fp16 [nb*h*w, kpad]
__global__ void im2col3x3_kernel(const float* __restrict__ x, int nb, int h, int w, int c, int kpad,
                                 __half* __restrict__ out) {
  size_t total = static_cast<size_t>(nb) * h * w * kpad;
  GRID_STRIDE(i, total) {
    int k = static_cast<int>(i % kpad);
    size_t row = i / kpad;
    float v = 0.f;
    if (k < 9 * c) {
      int tap = k / c, ch = k - tap * c;
      int ox = static_cast<int>(row % w);
      int oy = static_cast<int>((row / w) % h);
      int n = static_cast<int>(row / (static_cast<size_t>(w) * h));
      int iy = oy + tap / 3 - 1;
      int ix = ox + tap % 3 - 1;
      if (iy >= 0 && iy < h && ix >= 0 && ix < w) v = x[((static_cast<size_t>(n) * h + iy) * w + ix) * c + ch];
    }
    out[i] = __float2half_rn(v);
  }
}

__global__ void upsample2x_kernel(const float* __restrict__ x, int nb, int h, int w, int c, __half* __restrict__ out) {
  const int c4 = c / 4;
  size_t total = static_cast<size_t>(nb) * (2 * h) * (2 * w) * c4;
  GRID_STRIDE(i, total) {
    int cc = static_cast<int>(i % c4) * 4;
    size_t pix = i / c4;
    int ox = static_cast<int>(pix % (2 * w));
    int oy = static_cast<int>((pix / (2 * w)) % (2 * h));
    int n = static_cast<int>(pix / (static_cast<size_t>(4) * w * h));
    float4 v = *reinterpret_cast<const float4*>(x + ((static_cast<size_t>(n) * h + oy / 2) * w + ox / 2) * c + cc);
    __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&a);
    u.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(out + pix * c + cc) = u;
  }
}

__global__ void cast_f16_kernel(const float* __restrict__ x, size_t n, __half* __restrict__ out) {
  GRID_STRIDE(i, n) out[i] = __float2half_rn(x[i]);
}

// [batch, rows, ldx] (cols valid) -> [batch, cols, ldo] (rows valid). grid = (rows/32, cols/32, batch)
__global__ void transpose_f16_kernel(const __half* __restrict__ x, int rows, int cols, int ldx, __half* __restrict__ out,
                                     int ldo) {
  __shared__ __half tile[32][34];
  int b = blockIdx.z;
  int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int r = r0 + j, c = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (r < rows && c < cols) ? x[(static_cast<size_t>(b) * rows + r) * ldx + c] : __half(0.f);
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int c = c0 + j, r = r0 + threadIdx.x;
    if (c < cols && r < rows) out[(static_cast<size_t>(b) * cols + c) * ldo + r] = tile[threadIdx.x][j];
  }
}

struct StepCoef {
  float a_t, a_prev, sigma_t, sqrt_one_minus_a_t;
};
__global__ void sampler_step_kernel(const float* __restrict__ x, const float* __restrict__ eps2,
                                    const float* __restrict__ eps_cond, int guided, float scale, int order, const float* __restrict__ h1,
                                    const float* __restrict__ h2, const float* __restrict__ h3,
                                    const float* __restrict__ noise, StepCoef k, size_t n, float* __restrict__ x_prev,
                                    float* __restrict__ x_prev2, float* __restrict__ pred_x0,
                                    float* __restrict__ e_out) {
  // fp32 arithmetic in the reference's operation order (plms.py:185-186,199-216,224-232)
  const float sqrt_a_t = sqrtf(k.a_t);
  const float sqrt_a_prev = sqrtf(k.a_prev);
  const float dir_coef = sqrtf(__fsub_rn(__fsub_rn(1.0f, k.a_prev), __fmul_rn(k.sigma_t, k.sigma_t)));
  GRID_STRIDE(i, n) {
    float e_t;
    if (guided) {
      float eu = eps2[i], ec = eps_cond[i];
      e_t = __fadd_rn(eu, __fmul_rn(scale, __fsub_rn(ec, eu)));
    } else {
      e_t = eps2[i];
    }
    float ep;
    switch (order) {
      case 1: ep = __fdiv_rn(__fsub_rn(__fmul_rn(3.0f, e_t), h1[i]), 2.0f); break;
      case 2:
        ep = __fdiv_rn(__fadd_rn(__fsub_rn(__fmul_rn(23.0f, e_t), __fmul_rn(16.0f, h1[i])), __fmul_rn(5.0f, h2[i])), 12.0f);
        break;
      case 3:
        ep = __fdiv_rn(__fsub_rn(__fadd_rn(__fsub_rn(__fmul_rn(55.0f, e_t), __fmul_rn(59.0f, h1[i])), __fmul_rn(37.0f, h2[i])),
                                 __fmul_rn(9.0f, h3[i])), 24.0f);
        break;
      case 4: ep = __fdiv_rn(__fadd_rn(h1[i], e_t), 2.0f); break;
      default: ep = e_t; break;
    }
    float xv = x[i];
    // explicit rn ops: no FMA contraction, so the update matches the reference's separate fp32 tensor ops bit for bit
    float p0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(k.sqrt_one_minus_a_t, ep)), sqrt_a_t);
    float xp = __fadd_rn(__fmul_rn(sqrt_a_prev, p0), __fmul_rn(dir_coef, ep));
    if (noise) xp = __fadd_rn(xp, __fmul_rn(k.sigma_t, noise[i]));
    if (x_prev) x_prev[i] = xp;
    if (x_prev2) x_prev2[i] = xp;
    if (pred_x0) pred_x0[i] = p0;
    if (e_out) e_out[i] = e_t;
  }
}

// moments NHWC [nb*hw, 8] -> z NCHW [nb,4,hw]: (mean + exp(0.5*clamp(logvar,-30,20))*noise)*scale
__global__ void vae_sample_kernel(const float* __restrict__ moments, const float* __restrict__ noise, int nb, int hw,
                                  float scale_factor, float* __restrict__ z) {
  size_t total = static_cast<size_t>(nb) * 4 * hw;
  GRID_STRIDE(i, total) {
    int p = static_cast<int>(i % hw);
    int ch = static_cast<int>((i / hw) % 4);
    int n = static_cast<int>(i / (static_cast<size_t>(4) * hw));
    const float* m = moments + (static_cast<size_t>(n) * hw + p) * 8;
    float mean = m[ch];
    float logvar = fminf(fmaxf(m[4 + ch], -30.0f), 20.0f);
    float stdv = expf(0.5f * logvar);
    float eps = noise ? noise[i] : 0.f;
    z[i] = (mean + stdv * eps) * scale_factor;
  }
}

__global__ void to_uint8_kernel(const float* __restrict__ x, size_t n, uint8_t* __restrict__ out) {
  GRID_STRIDE(i, n) {
    float v = fminf(fmaxf((x[i] + 1.0f) * 0.5f, 0.0f), 1.0f);
    out[i] = static_cast<uint8_t>(255.0f * v);  // matches (255. * x).astype(uint8) truncation, txt2img.py:322-323
  }
}

// DPM-Solver++ multistep update in data-prediction form (dpm_solver.py:386-399, 504-533, 755-789), fp32 in the
// reference's operation order: m0 = (x - sigma_s e) / alpha_s; order 1: x_t = c_x x - c_m m0;
// order 2: x_t = c_x x - c_m m0 - (0.5 c_m) * (inv_r0 (m0 - m_prev))
__global__ void dpm_solver_step_kernel(const float* __restrict__ x, const float* __restrict__ eps2,
                                       const float* __restrict__ eps_cond, int guided, float scale, float sigma_s, float alpha_s, int order,
                                       const float* __restrict__ m_prev, float c_x, float c_m, float inv_r0, size_t n,
                                       float* __restrict__ m_out, float* __restrict__ x_out,
                                       float* __restrict__ x_out2) {
  const float half_c_m = __fmul_rn(0.5f, c_m);
  GRID_STRIDE(i, n) {
    float e;
    if (guided) {
      float eu = eps2[i], ec = eps_cond[i];
      e = __fadd_rn(eu, __fmul_rn(scale, __fsub_rn(ec, eu)));
    } else {
      e = eps2[i];
    }
    const float xv = x[i];
    const float m0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(sigma_s, e)), alpha_s);
    float xt = __fsub_rn(__fmul_rn(c_x, xv), __fmul_rn(c_m, m0));
    if (order == 2) xt = __fsub_rn(xt, __fmul_rn(half_c_m, __fmul_rn(inv_r0, __fsub_rn(m0, m_prev[i]))));
    if (m_out) m_out[i] = m0;
    x_out[i] = xt;
    if (x_out2) x_out2[i] = xt;
  }
}

// inpainting blend (plms.py:147-150, ddim.py:144-147): img = img_orig * mask + (1 - mask) * img; the mask is
// [b, 1, h, w] (broadcast over channels) or [b, c, h, w]
__global__ void mask_blend_kernel(const float* __restrict__ img_orig, const float* __restrict__ mask, int bcast,
                                  size_t n, size_t chw, size_t hw, float* __restrict__ img, float* __restrict__ img2) {
  GRID_STRIDE(i, n) {
    const size_t mi = bcast ? (i / chw) * hw + (i % hw) : i;
    const float m = mask[mi];
    const float v = __fadd_rn(__fmul_rn(img_orig[i], m), __fmul_rn(__fsub_rn(1.0f, m), img[i]));
    img[i] = v;
    if (img2) img2[i] = v;
  }
}

__global__ void axpby2_kernel(const float* __restrict__ x, const float* __restrict__ y, float a, float b, size_t n,
                              float* __restrict__ out) {
  GRID_STRIDE(i, n) out[i] = __fadd_rn(__fmul_rn(a, x[i]), __fmul_rn(b, y[i]));
}

__global__ void axpby_kernel(const float* __restrict__ x, float a, float b, size_t n, float* __restrict__ out) {
  GRID_STRIDE(i, n) out[i] = a * x[i] + b;
}

// per-pixel small channel mix (1x1 conv with <= 8 channels, fp32): out[p, j] = alpha * sum_c x[p, c] w[j, c] + b[j]
__global__ void pointwise_small_kernel(const float* __restrict__ x, size_t npix, int cin, int cout,
                                       const float* __restrict__ w, const float* __restrict__ b, float alpha,
                                       float* __restrict__ out) {
  GRID_STRIDE(i, npix * cout) {
    size_t p = i / cout;
    int j = static_cast<int>(i - p * cout);
    float acc = 0.f;
    for (int c = 0; c < cin; ++c) acc = fmaf(x[p * cin + c] * alpha, w[j * cin + c], acc);
    out[i] = acc + (b ? b[j] : 0.f);
  }
}

// CLIP embeddings: out[b*n + i, :] = tok[ids[b, i], :] + pos[i, :]   (fp32)
__global__ void embed_tokens_kernel(const long long* __restrict__ ids, int rows, int n_ctx, int dim, int vocab,
                                    const float* __restrict__ tok, const float* __restrict__ pos,
                                    float* __restrict__ out) {
  GRID_STRIDE(i, static_cast<size_t>(rows) * dim) {
    int r = static_cast<int>(i / dim), c = static_cast<int>(i % dim);
    long long id = ids[r];
    if (id < 0) id = 0;
    if (id >= vocab) id = vocab - 1;
    out[i] = tok[static_cast<size_t>(id) * dim + c] + pos[static_cast<size_t>(r % n_ctx) * dim + c];
  }
}

}  // namespace sdb

using namespace sdb;
#define ST static_cast<cudaStream_t>(stream)

extern "C" int sdb_nchw_to_nhwc(const float* x, int32_t nb, int32_t c, int32_t hw, float* out_f32, void* out_f16,
                                sdb_stream_t stream) {
  SDB_REC(sdb_nchw_to_nhwc(x, nb, c, hw, out_f32, out_f16, s_));
  SDB_CHECK(x && (out_f32 || out_f16), "sdb_nchw_to_nhwc: null pointer");
  dim3 grid((hw + 31) / 32, (c + 31) / 32, nb), block(32, 8);
  nchw_to_nhwc_kernel<<<grid, block, 0, ST>>>(x, c, hw, out_f32, static_cast<__half*>(out_f16));
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_nhwc_to_nchw(const float* x, int32_t nb, int32_t c, int32_t hw, float* out, sdb_stream_t stream) {
  SDB_REC(sdb_nhwc_to_nchw(x, nb, c, hw, out, s_));
  SDB_CHECK(x && out, "sdb_nhwc_to_nchw: null pointer");
  dim3 grid((hw + 31) / 32, (c + 31) / 32, nb), block(32, 8);
  nhwc_to_nchw_kernel<<<grid, block, 0, ST>>>(x, c, hw, out);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_im2col3x3(const float* x, int32_t nb, int32_t h, int32_t w, int32_t c, int32_t kpad, void* out_f16,
                             sdb_stream_t stream) {
  SDB_REC(sdb_im2col3x3(x, nb, h, w, c, kpad, out_f16, s_));
  SDB_CHECK(x && out_f16 && kpad >= 9 * c && kpad % 64 == 0, "sdb_im2col3x3: bad arguments (kpad=%d c=%d)", kpad, c);
  size_t total = static_cast<size_t>(nb) * h * w * kpad;
  im2col3x3_kernel<<<grid_for(total), 256, 0, ST>>>(x, nb, h, w, c, kpad, static_cast<__half*>(out_f16));
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_upsample2x(const float* x, int32_t nb, int32_t h, int32_t w, int32_t c, void* out_f16,
                              sdb_stream_t stream) {
  SDB_REC(sdb_upsample2x(x, nb, h, w, c, out_f16, s_));
  SDB_CHECK(x && out_f16 && c % 4 == 0, "sdb_upsample2x: bad arguments");
  size_t total = static_cast<size_t>(nb) * 4 * h * w * (c / 4);
  upsample2x_kernel<<<grid_for(total), 256, 0, ST>>>(x, nb, h, w, c, static_cast<__half*>(out_f16));
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_cast_f16(const float* x, int64_t n, void* out_f16, sdb_stream_t stream) {
  SDB_REC(sdb_cast_f16(x, n, out_f16, s_));
  SDB_CHECK(x && out_f16 && n >= 0, "sdb_cast_f16: bad arguments");
  cast_f16_kernel<<<grid_for(n), 256, 0, ST>>>(x, static_cast<size_t>(n), static_cast<__half*>(out_f16));
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_transpose_f16(const void* x, int32_t batch, int32_t rows, int32_t cols, int32_t ldx, void* out,
                                 int32_t ldo, sdb_stream_t stream) {
  SDB_REC(sdb_transpose_f16(x, batch, rows, cols, ldx, out, ldo, s_));
  SDB_CHECK(x && out && ldx >= cols && ldo >= rows, "sdb_transpose_f16: bad arguments");
  dim3 grid((rows + 31) / 32, (cols + 31) / 32, batch), block(32, 8);
  transpose_f16_kernel<<<grid, block, 0, ST>>>(static_cast<const __half*>(x), rows, cols, ldx,
                                               static_cast<__half*>(out), ldo);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_sampler_step(const float* x, const float* eps2, const float* eps_cond, int32_t guided, float scale,
                                int32_t order,
                                const float* h1, const float* h2, const float* h3, const float* noise, float a_t,
                                float a_prev, float sigma_t, float sqrt_one_minus_a_t, int64_t n, float* x_prev,
                                float* x_prev2, float* pred_x0, float* e_out, sdb_stream_t stream) {
  SDB_REC(sdb_sampler_step(x, eps2, eps_cond, guided, scale, order, h1, h2, h3, noise, a_t, a_prev, sigma_t, sqrt_one_minus_a_t, n, x_prev, x_prev2, pred_x0, e_out, s_));
  SDB_CHECK(x && eps2 && n > 0, "sdb_sampler_step: bad arguments");
  SDB_CHECK(order >= 0 && order <= 4, "sdb_sampler_step: order %d", order);
  SDB_CHECK((order == 0) || h1, "sdb_sampler_step: missing history");
  StepCoef k{a_t, a_prev, sigma_t, sqrt_one_minus_a_t};
  if (!eps_cond) eps_cond = eps2 + n;   // [e_uncond; e_cond] contiguous
  sampler_step_kernel<<<grid_for(n), 256, 0, ST>>>(x, eps2, eps_cond, guided, scale, order, h1, h2, h3, noise, k,
                                                   static_cast<size_t>(n), x_prev, x_prev2, pred_x0, e_out);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_dpm_solver_step(const float* x, const float* eps2, const float* eps_cond, int32_t guided, float scale,
                                   float sigma_s,
                                   float alpha_s, int32_t order, const float* m_prev, float c_x, float c_m,
                                   float inv_r0, int64_t n, float* m_out, float* x_out, float* x_out2,
                                   sdb_stream_t stream) {
  SDB_REC(sdb_dpm_solver_step(x, eps2, eps_cond, guided, scale, sigma_s, alpha_s, order, m_prev, c_x, c_m, inv_r0, n, m_out, x_out, x_out2, s_));
  SDB_CHECK(x && eps2 && x_out && n > 0, "sdb_dpm_solver_step: bad arguments");
  SDB_CHECK(order == 1 || (order == 2 && m_prev), "sdb_dpm_solver_step: order %d (2 needs the previous prediction)", order);
  if (!eps_cond) eps_cond = eps2 + n;
  dpm_solver_step_kernel<<<grid_for(n), 256, 0, ST>>>(x, eps2, eps_cond, guided, scale, sigma_s, alpha_s, order, m_prev, c_x, c_m,
                                                      inv_r0, static_cast<size_t>(n), m_out, x_out, x_out2);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_mask_blend(const float* img_orig, const float* mask, int32_t mask_channels, int32_t nb, int32_t c,
                              int64_t hw, float* img, float* img2, sdb_stream_t stream) {
  SDB_REC(sdb_mask_blend(img_orig, mask, mask_channels, nb, c, hw, img, img2, s_));
  SDB_CHECK(img_orig && mask && img && nb > 0 && c > 0 && hw > 0, "sdb_mask_blend: bad arguments");
  SDB_CHECK(mask_channels == 1 || mask_channels == c, "sdb_mask_blend: mask has %d channels, latent %d", mask_channels, c);
  const size_t n = static_cast<size_t>(nb) * c * hw;
  mask_blend_kernel<<<grid_for(n), 256, 0, ST>>>(img_orig, mask, mask_channels == 1 ? 1 : 0, n,
                                                 static_cast<size_t>(c) * hw, static_cast<size_t>(hw), img, img2);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_vae_sample(const float* moments, const float* noise_nchw, int32_t nb, int32_t hw,
                              float scale_factor, float* z_nchw, sdb_stream_t stream) {
  SDB_REC(sdb_vae_sample(moments, noise_nchw, nb, hw, scale_factor, z_nchw, s_));
  SDB_CHECK(moments && z_nchw, "sdb_vae_sample: null pointer");
  vae_sample_kernel<<<grid_for(static_cast<size_t>(nb) * 4 * hw), 256, 0, ST>>>(moments, noise_nchw, nb, hw,
                                                                                scale_factor, z_nchw);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_to_uint8(const float* x, int64_t n, uint8_t* out, sdb_stream_t stream) {
  SDB_REC(sdb_to_uint8(x, n, out, s_));
  SDB_CHECK(x && out, "sdb_to_uint8: null pointer");
  to_uint8_kernel<<<grid_for(n), 256, 0, ST>>>(x, static_cast<size_t>(n), out);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_axpby2(const float* x, const float* y, float a, float b, int64_t n, float* out,
                          sdb_stream_t stream) {
  SDB_REC(sdb_axpby2(x, y, a, b, n, out, s_));
  SDB_CHECK(x && y && out, "sdb_axpby2: null pointer");
  axpby2_kernel<<<grid_for(n), 256, 0, ST>>>(x, y, a, b, static_cast<size_t>(n), out);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_axpby(const float* x, float a, float b, int64_t n, float* out, sdb_stream_t stream) {
  SDB_REC(sdb_axpby(x, a, b, n, out, s_));
  SDB_CHECK(x && out, "sdb_axpby: null pointer");
  axpby_kernel<<<grid_for(n), 256, 0, ST>>>(x, a, b, static_cast<size_t>(n), out);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_pointwise_small(const float* x, int64_t npix, int32_t cin, int32_t cout, const float* w,
                                   const float* b, float alpha, float* out, sdb_stream_t stream) {
  SDB_REC(sdb_pointwise_small(x, npix, cin, cout, w, b, alpha, out, s_));
  SDB_CHECK(x && w && out && cin > 0 && cin <= 16 && cout > 0 && cout <= 16, "sdb_pointwise_small: bad arguments");
  pointwise_small_kernel<<<grid_for(static_cast<size_t>(npix) * cout), 256, 0, ST>>>(
      x, static_cast<size_t>(npix), cin, cout, w, b, alpha, out);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" int sdb_embed_tokens(const int64_t* ids, int32_t rows, int32_t n_ctx, int32_t dim, int32_t vocab,
                                const float* tok, const float* pos, float* out, sdb_stream_t stream) {
  SDB_REC(sdb_embed_tokens(ids, rows, n_ctx, dim, vocab, tok, pos, out, s_));
  SDB_CHECK(ids && tok && pos && out, "sdb_embed_tokens: null pointer");
  embed_tokens_kernel<<<grid_for(static_cast<size_t>(rows) * dim), 256, 0, ST>>>(
      reinterpret_cast<const long long*>(ids), rows, n_ctx, dim, vocab, tok, pos, out);
  SDB_LAUNCH_CHECK();
  return 0;
}
extern "C" const char* sdb_last_error(void) { return sdb::last_error(); }
extern "C" int sdb_version(void) { return 101; }
extern "C" int sdb_sm_count(void) { return sdb::sm_count(); }
extern "C" long long sdb_launch_count(void) { return sdb::launch_count(); }
extern "C" long long sdb_debug_trace(void* buf, int64_t n_words) {
  long long used = sdb::trace_used();
  sdb::set_trace(buf, n_words);
  return used;
}
