// Handle-level entry points of the C ABI: a maintainer who binds libsdb200.so gets the ENGINE - one call per UNet
// evaluation (sdb_unet_forward) and one per sampling trajectory (sdb_sample_plms) - not a bag of kernels plus a host
// scheduler to rewrite.
//
//   sdb_plan      : an ordered list of sdb_* launches with their arguments (descriptors copied by value), recorded while
//                   the host side walks the model once (sdb_plan_begin .. sdb_plan_end; the calls still execute). The
//                   plan owns a CUDA graph of the sequence, built on first launch by replaying the list under stream
//                   capture on a private stream; afterwards one cudaGraphLaunch per evaluation. All pointers are the
//                   caller's static buffers (weights, workspaces, I/O): they must outlive the plan.
//   sdb_unet      : plan of one guided UNet evaluation + its static x / t / eps buffers
//                   (replaces the call chain sampler -> LatentDiffusion.apply_model -> DiffusionWrapper -> UNetModel.forward,
//                   ldm/models/diffusion/ddpm.py:891-992,1393-1421; ldm/modules/diffusionmodules/openaimodel.py:710-742)
//   sdb_sample_plms: the whole PLMS trajectory (ldm/models/diffusion/plms.py:98-236: first step pseudo improved Euler
//                   with a second evaluation, then Adams-Bashforth orders 2-4) as unet launches + fused step kernels,
//                   with the schedule passed as plain host arrays.
#include "../../include/sdb200.h"
#include "host.h"

#include <functional>
#include <new>
#include <vector>

struct sdb_plan {
  std::vector<std::function<int(cudaStream_t)>> ops;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  cudaStream_t capture_stream = nullptr;
  bool closed = false;
};

struct sdb_unet {
  sdb_plan* plan;
  float* x;     // static input  [n, c_in, h, w] the plan's first kernel reads
  float* t;     // static timesteps [n]
  float* eps;   // static output [n, c_out, h, w] the plan's last kernel writes
  int n, c_in, c_out, h, w;
};

namespace sdb {

static thread_local sdb_plan* g_rec = nullptr;

bool plan_recording() { return g_rec != nullptr; }
void plan_record(std::function<int(cudaStream_t)> fn) {
  if (g_rec) g_rec->ops.push_back(std::move(fn));
}

__global__ void fill_f32_kernel(float* p, int n, float v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

static int run_ops(sdb_plan* p, cudaStream_t st) {
  sdb_plan* keep = g_rec;
  g_rec = nullptr;   // replaying must not record
  int rc = 0;
  for (auto& op : p->ops) {
    rc = op(st);
    if (rc) break;
  }
  g_rec = keep;
  return rc;
}

}  // namespace sdb

using namespace sdb;

extern "C" int sdb_plan_begin(sdb_plan** out) {
  SDB_CHECK(out != nullptr, "sdb_plan_begin: null argument");
  SDB_CHECK(g_rec == nullptr, "sdb_plan_begin: a plan is already being recorded on this thread");
  sdb_plan* p = new (std::nothrow) sdb_plan();
  SDB_CHECK(p != nullptr, "sdb_plan_begin: out of memory");
  g_rec = p;
  *out = p;
  return 0;
}

extern "C" int sdb_plan_end(sdb_plan* p) {
  SDB_CHECK(p != nullptr && g_rec == p, "sdb_plan_end: this plan is not being recorded");
  g_rec = nullptr;
  p->closed = true;
  return 0;
}

extern "C" int sdb_plan_size(const sdb_plan* p) { return p ? static_cast<int>(p->ops.size()) : -1; }

extern "C" int sdb_plan_launch(sdb_plan* p, sdb_stream_t stream) {
  SDB_CHECK(p && p->closed, "sdb_plan_launch: plan not recorded");
  SDB_CHECK(!p->ops.empty(), "sdb_plan_launch: empty plan");
  if (!p->exec) {
    // capture the recorded sequence once, on a private stream (the caller's may be the legacy default stream)
    if (!p->capture_stream) SDB_CUDA(cudaStreamCreateWithFlags(&p->capture_stream, cudaStreamNonBlocking));
    SDB_CUDA(cudaStreamBeginCapture(p->capture_stream, cudaStreamCaptureModeThreadLocal));
    const int rc = run_ops(p, p->capture_stream);
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(p->capture_stream, &g);
    if (rc) {
      if (g) cudaGraphDestroy(g);
      return rc;
    }
    SDB_CUDA(e);
    p->graph = g;
    SDB_CUDA(cudaGraphInstantiate(&p->exec, p->graph, 0));
  }
  SDB_CUDA(cudaGraphLaunch(p->exec, static_cast<cudaStream_t>(stream)));
  return 0;
}

extern "C" int sdb_plan_destroy(sdb_plan* p) {
  if (!p) return 0;
  if (g_rec == p) g_rec = nullptr;
  if (p->exec) cudaGraphExecDestroy(p->exec);
  if (p->graph) cudaGraphDestroy(p->graph);
  if (p->capture_stream) cudaStreamDestroy(p->capture_stream);
  delete p;
  return 0;
}

extern "C" int sdb_fill_f32(float* x, int64_t n, float value, sdb_stream_t stream) {
  SDB_CHECK(x != nullptr && n > 0 && n < (1LL << 31), "sdb_fill_f32: bad arguments");
  if (plan_recording()) plan_record([=](cudaStream_t s) { return sdb_fill_f32(x, n, value, s); });
  fill_f32_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<int>(n),
                                                                                                   value);
  SDB_LAUNCH_CHECK();
  return 0;
}

extern "C" int sdb_unet_create(sdb_plan* plan, float* x_static, float* t_static, float* eps_static, int32_t n,
                               int32_t c_in, int32_t c_out, int32_t h, int32_t w, sdb_unet** out) {
  SDB_CHECK(plan && plan->closed && !plan->ops.empty(), "sdb_unet_create: the plan has not been recorded");
  SDB_CHECK(x_static && t_static && eps_static && out, "sdb_unet_create: null pointer");
  SDB_CHECK(n > 0 && c_in > 0 && c_out > 0 && h > 0 && w > 0, "sdb_unet_create: bad dims");
  sdb_unet* u = new (std::nothrow) sdb_unet{plan, x_static, t_static, eps_static, n, c_in, c_out, h, w};
  SDB_CHECK(u != nullptr, "sdb_unet_create: out of memory");
  *out = u;
  return 0;
}

extern "C" int sdb_unet_destroy(sdb_unet* u) {
  delete u;
  return 0;
}

extern "C" int sdb_unet_forward(sdb_unet* u, const float* x, const float* t, float* eps, sdb_stream_t stream) {
  SDB_CHECK(u != nullptr, "sdb_unet_forward: null handle");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t nx = static_cast<size_t>(u->n) * u->c_in * u->h * u->w, ne = static_cast<size_t>(u->n) * u->c_out * u->h * u->w;
  if (x && x != u->x) SDB_CUDA(cudaMemcpyAsync(u->x, x, nx * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (t && t != u->t) SDB_CUDA(cudaMemcpyAsync(u->t, t, u->n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (int rc = sdb_plan_launch(u->plan, stream)) return rc;
  if (eps && eps != u->eps) SDB_CUDA(cudaMemcpyAsync(eps, u->eps, ne * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}

extern "C" int sdb_sample_plms(const sdb_plms_desc* d, sdb_stream_t stream) {
  SDB_CHECK(d && d->unet && d->x && d->work && d->timesteps && d->alphas && d->alphas_prev && d->sqrt_one_minus_alphas,
            "sdb_sample_plms: null pointer");
  sdb_unet* u = d->unet;
  const int rep = d->guided ? 2 : 1;
  SDB_CHECK(u->n == rep * d->batch, "sdb_sample_plms: the UNet plan evaluates %d samples, need %d", u->n, rep * d->batch);
  SDB_CHECK(u->c_in == u->c_out, "sdb_sample_plms: eps and x must have the same shape");
  SDB_CHECK(d->n_steps >= 1, "sdb_sample_plms: n_steps");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t per = static_cast<int64_t>(d->batch) * u->c_in * u->h * u->w;   // elements of one (un-doubled) latent batch
  // workspace: 4 eps history slots + pred_x0 + the first step's intermediate latent (doubled)
  float* hist[4] = {d->work, d->work + per, d->work + 2 * per, d->work + 3 * per};
  float* pred_x0 = d->work + 4 * per;
  float* xp = d->work + 5 * per;              // [rep * per]
  float* xa = u->x;                           // the latent ping-pongs between the plan's static input buffer ...
  float* xb = d->work + (5 + rep) * per;      // ... and this one ([rep * per]). It starts in xb: the first step evaluates
                                              // the UNet twice and must still hold x_t afterwards
  SDB_CUDA(cudaMemcpyAsync(xb, d->x, per * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (rep == 2) SDB_CUDA(cudaMemcpyAsync(xb + per, d->x, per * sizeof(float), cudaMemcpyDeviceToDevice, st));
  int n_hist = 0, head = 0;   // ring of the last <= 3 eps: hist[(head - 1 - j) & 3] is the j-th most recent
  float* cur = xb;
  float* nxt = xa;
  auto eval = [&](const float* xin, float tval) -> int {
    if (int rc = sdb_fill_f32(u->t, u->n, tval, stream)) return rc;
    return sdb_unet_forward(u, xin, nullptr, nullptr, stream);
  };
  auto step = [&](const float* x2, int index, int order, const float* h0, const float* h1, const float* h2, float* x_prev,
                  float* e_out) -> int {
    return sdb_sampler_step(x2, u->eps, nullptr, d->guided, d->scale, order, h0, h1, h2, nullptr, d->alphas[index],
                            d->alphas_prev[index], d->sigmas ? d->sigmas[index] : 0.f, d->sqrt_one_minus_alphas[index], per,
                            x_prev, rep == 2 ? x_prev + per : nullptr, pred_x0, e_out, stream);
  };
  for (int i = 0; i < d->n_steps; ++i) {
    const int index = d->n_steps - 1 - i;                     // schedule arrays are indexed like the reference's ddim_* arrays
    const float t_cur = d->timesteps[index];
    const float t_next = d->timesteps[index > 0 ? index - 1 : 0];
    if (int rc = eval(cur, t_cur)) return rc;
    float* e_t = hist[head & 3];
    if (n_hist == 0) {
      // pseudo improved Euler (plms.py:213-217): x' from e_t alone, a second evaluation at t_next, e' = (e_t + e_t_next) / 2
      if (int rc = step(cur, index, 0, nullptr, nullptr, nullptr, xp, e_t)) return rc;
      if (int rc = eval(xp, t_next)) return rc;
      if (int rc = step(cur, index, 4, e_t, nullptr, nullptr, nxt, nullptr)) return rc;
    } else {
      const int order = n_hist < 3 ? n_hist : 3;
      const float* h0 = hist[(head - 1) & 3];
      const float* h1 = order > 1 ? hist[(head - 2) & 3] : nullptr;
      const float* h2 = order > 2 ? hist[(head - 3) & 3] : nullptr;
      if (int rc = step(cur, index, order, h0, h1, h2, nxt, e_t)) return rc;
    }
    ++head;
    if (n_hist < 3) ++n_hist;
    float* tmp = cur;
    cur = nxt;
    nxt = tmp;
  }
  if (d->x_out) SDB_CUDA(cudaMemcpyAsync(d->x_out, cur, per * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (d->pred_x0_out) SDB_CUDA(cudaMemcpyAsync(d->pred_x0_out, pred_x0, per * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}
