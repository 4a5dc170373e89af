// C-ABI entry points (include/sgp.h): context, multi-GPU plumbing, the statistics pipeline.
#include "sgp_internal.h"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>

namespace sgp {

static thread_local std::string g_create_err;

// NCCL is resolved lazily with dlopen instead of being a link-time dependency: a host process that also
// loads PyTorch already carries torch's own libnccl.so.2, and two different NCCL builds under one soname
// cannot coexist.  dlopen("libnccl.so.2") returns the copy that is already mapped, else the system one.
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};
static NcclApi& nccl() {
  static NcclApi api = [] {
    NcclApi a;
    void* h = dlopen("libnccl.so.2", RTLD_LAZY | RTLD_LOCAL);
    if (!h) h = dlopen("libnccl.so", RTLD_LAZY | RTLD_LOCAL);
    if (!h) return a;
    a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
    a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
    a.AllReduce = reinterpret_cast<decltype(a.AllReduce)>(dlsym(h, "ncclAllReduce"));
    a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
    a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
    a.ok = a.GetUniqueId && a.CommInitRank && a.AllReduce && a.CommDestroy && a.GetErrorString;
    return a;
  }();
  return api;
}

int fail(Ctx* c, int code, const std::string& msg) {
  if (c) {
    c->err = msg;
    if (code == SGP_E_CUDA && c->i8_pm_host && c->i8_pm_host[0] != 0) {
      const int* pm = c->i8_pm_host;            // int8 kernel post-mortem: first wait that made no progress for ~1 s
      long long unit;
      std::memcpy(&unit, pm + 4, sizeof(unit));
      c->err += " [kmn_gram_i8 post-mortem: wait site " + std::to_string(pm[0]) + " block (" + std::to_string(pm[1]) + "," +
                std::to_string(pm[2]) + ") warp " + std::to_string(pm[3]) + " unit " + std::to_string(unit) + " a=" +
                std::to_string(static_cast<unsigned>(pm[6])) + " b=" + std::to_string(static_cast<unsigned>(pm[7])) + "]";
    }
  } else {
    g_create_err = msg;
  }
  return code;
}

static void free_active_set(Ctx* c) {
  cudaFree(c->dZ); cudaFree(c->dZs); cudaFree(c->dBeta); cudaFree(c->dGb);
  cudaFree(c->dMagicVec); cudaFree(c->dMagicMat);
  cudaFree(c->dI8Scale); cudaFree(c->dI8Centre); cudaFree(c->dI8Flags); cudaFree(c->dI8Zt); cudaFree(c->dI8NormSum);
  cudaFree(c->dI8Zd); cudaFree(c->dI8DScale); c->dI8Zd = nullptr; c->dI8DScale = nullptr; c->i8_direct_ok = false;
  c->i8d_zd_bytes = c->i8d_sc_bytes = 0; c->i8d_prepared = false;
  c->dI8NormSum = nullptr;
  c->dZ = c->dZs = c->dBeta = c->dGb = c->dMagicVec = c->dMagicMat = nullptr;
  c->dI8Scale = c->dI8Centre = nullptr; c->dI8Flags = nullptr; c->dI8Zt = nullptr; c->i8_ok = false;
}

static int ensure_partials(Ctx* c, int n_slices) {
  const size_t gb = static_cast<size_t>(n_slices) * c->m_pad * c->m_pad * sizeof(double);
  const size_t bb = static_cast<size_t>(n_slices) * c->m_pad * sizeof(double);
  if (gb > c->gpart_bytes) {
    cudaFree(c->dGpart); c->dGpart = nullptr; c->gpart_bytes = 0;
    SGP_CUDA(c, cudaMalloc(&c->dGpart, gb));
    c->gpart_bytes = gb;
  }
  if (bb > c->bpart_bytes) {
    cudaFree(c->dBpart); c->dBpart = nullptr; c->bpart_bytes = 0;
    SGP_CUDA(c, cudaMalloc(&c->dBpart, bb));
    c->bpart_bytes = bb;
  }
  return SGP_OK;
}

// Device side of the direct-distance mode for the current begin() window: per-term scales + centre, active-set tiles
int direct_prepare(Ctx* c) {
  if (c->i8d_prepared) return SGP_OK;
  const int dpad4 = c->i8_dpad4;
  const size_t zd_bytes = static_cast<size_t>(c->m_pad / kTile) * c->kf.n_terms * kTile * dpad4 * sizeof(float);
  const size_t sc_bytes = c->i8d_sc.size() * 8;
  if (zd_bytes > c->i8d_zd_bytes || sc_bytes > c->i8d_sc_bytes || !c->dI8Zd) {
    cudaFree(c->dI8Zd); cudaFree(c->dI8DScale); c->dI8Zd = nullptr; c->dI8DScale = nullptr;
    c->i8d_zd_bytes = c->i8d_sc_bytes = 0;
    SGP_CUDA(c, cudaMalloc(&c->dI8Zd, zd_bytes));
    SGP_CUDA(c, cudaMalloc(&c->dI8DScale, sc_bytes));
    c->i8d_zd_bytes = zd_bytes; c->i8d_sc_bytes = sc_bytes;
  }
  SGP_CUDA(c, cudaMemcpyAsync(c->dI8DScale, c->i8d_sc.data(), sc_bytes, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, launch_i8_prep_active_direct(c->dI8Zd, c->dZ, c->m, c->m_pad, c->d, dpad4, c->kf.n_terms, c->dI8DScale,
                                           c->dI8DScale + static_cast<size_t>(kMaxTerms) * dpad4, c->dI8Flags,
                                           c->i8_direct_r2max, c->stream));
  c->launches += 1;
  c->i8d_prepared = true;
  return SGP_OK;
}

// One fused-kernel launch over n device-resident points + the deterministic slice reduction.
static int launch_stats(Ctx* c, const void* dX, int x_is_f32, const double* dy, long long n, long long n_call,
                        bool first_of_call) {
  // n: points of this launch; n_call: points of the whole accumulate call.  AUTO decides per CALL -- the size gate
  // looks at n_call and the magnitude gate at the first chunk -- so the chunks of one shard never mix kernels (and
  // only the first chunk pays the device->host round trip of the gate)
  if (n <= 0) return SGP_OK;
  const int nt1 = c->m_pad / kTile;
  const int ntiles = nt1 * (nt1 + 1) / 2;
  int n_slices = c->num_sms / ntiles;            // fp64 kernel: fill the SMs with tiles x point-slices
  if (n_slices < 1) n_slices = 1;
  const long long blocks = (n + 15) / 16;
  if (n_slices > blocks) n_slices = static_cast<int>(blocks);
  // int8 kernel: cooperative launches of whole tile columns (all CTAs of a launch are co-resident)
  I8Launch plan[64];
  int n_plan = 0, plan_slices = 1;
  if ((c->i8_ok || c->i8_direct_ok) && c->i8_impl == 1) {
    n_plan = i8_plan(c->m_pad, c->num_sms, (n + 63) / 64, plan, 64);
    for (int i = 0; i < n_plan; ++i) plan_slices = plan[i].n_slices > plan_slices ? plan[i].n_slices : plan_slices;
  }
  int rc = ensure_partials(c, n_slices > plan_slices ? n_slices : plan_slices);
  if (rc != SGP_OK) return rc;

  GramParams p{};
  p.X = dX; p.y = dy; p.n = n; p.x_is_f32 = x_is_f32;
  p.d = c->d; p.dpad = c->dpad; p.m = c->m; p.m_pad = c->m_pad;
  p.n_terms = c->kf.n_terms;
  for (int t = 0; t < kMaxTerms; ++t) p.scale[t] = c->kf.scale[t];
  p.Zs = c->dZs; p.beta = c->dBeta;
  p.Gpart = c->dGpart; p.bpart = c->dBpart;
  p.n_slices = n_slices; p.n_tiles_1d = nt1;

  // AUTO: the tcgen05 int8 kernel inside its measured parity envelope -- accumulate calls of >= 32768 points (posterior
  // mean within 1.1e-6 .. 2.4e-6 of the all-fp64 kernel for N = 16k .. 4M: profiles/r01_i8_scaling.txt,
  // profiles/r02n_i8_small_shards.txt; the limit is the two dropped low-order digit products, tools/i8_error_model.py,
  // and does not grow towards small N) and small scaled norms (gate below).  Smaller calls stay on the fp64 DMMA kernel
  // (2e-7), which needs < 2 ms at that size.
  // Path of this launch: 0 = fp64 DMMA kernel, 1 = int8 Gram with tensor-core distances (one term, d <= 32, benign norms),
  // 2 = int8 Gram with direct fp32 distances (up to 4 terms, d <= 72; AUTO: same magnitude budget as path 1).
  const bool tensor_ok = c->i8_ok, direct_ok = c->i8_direct_ok && c->i8_impl == 1 && n_plan > 0;
  int path = 0;
  if (c->precision == SGP_PREC_I8) {
    if (tensor_ok) path = 1;
    else if (direct_ok) path = 2;
    else return fail(c, SGP_E_BADARG, "SGP_PREC_I8 needs a kernel with 1..4 non-Eye terms and n_terms * d <= 72 "
                                      "(tensor-core distances: exactly one term and d <= 32)");
  } else if (c->precision == SGP_PREC_I8_DIRECT) {
    if (!direct_ok) return fail(c, SGP_E_BADARG, "SGP_PREC_I8_DIRECT needs a kernel with 1..4 non-Eye terms and n_terms * d <= 72");
    path = 2;
  } else if (c->precision == SGP_PREC_AUTO && n_call >= kAutoI8MinPoints) {
    path = tensor_ok ? 1 : (direct_ok ? 2 : 0);
    if (!first_of_call) path = c->call_path;
  }
  bool use_i8 = (path == 1);
  if (use_i8 && c->i8_impl == 1 && n_plan <= 0) {
    if (c->precision == SGP_PREC_I8) return fail(c, SGP_E_BADARG, "active set too large for the int8 kernel's launch plan");
    use_i8 = false; path = 0;
  }
  if (path != 0) {
    const size_t yb = static_cast<size_t>((n + 63) / 64) * 64 * sizeof(float);
    if (yb > c->i8_ys_bytes) {
      cudaFree(c->dI8Ys); c->dI8Ys = nullptr; c->i8_ys_bytes = 0;
      SGP_CUDA(c, cudaMalloc(&c->dI8Ys, yb));
      c->i8_ys_bytes = yb;
    }
    if (c->i8_impl == 1) {
      rc = ctx_scratch(c, c->i8_share, i8_share_bytes(c->m_pad, plan_slices));
      if (rc != SGP_OK) return rc;
    }
  }
  if (use_i8) {
    const int nch = i8_nchunks(c->d);
    const size_t xb = i8_points_scratch_bytes(n, nch);
    if (xb > c->i8_xt_bytes) {
      cudaFree(c->dI8Xt); c->dI8Xt = nullptr; c->i8_xt_bytes = 0;
      SGP_CUDA(c, cudaMalloc(&c->dI8Xt, xb));
      c->i8_xt_bytes = xb;
    }
    const bool gate = (c->precision == SGP_PREC_AUTO) && first_of_call;
    // the scaled squared norms of EVERY chunk are summed on the device (dI8NormSum[0]: whole begin..finish window,
    // checked against the budget at finish so that an unrepresentative first chunk cannot silently degrade the
    // statistics; dI8NormSum[1]: this call's first chunk, read back here for the kernel choice)
    if (gate) SGP_CUDA(c, cudaMemsetAsync(c->dI8NormSum + 1, 0, sizeof(double), c->stream));
    SGP_CUDA(c, launch_i8_prep_points(c->dI8Xt, c->dI8Ys, dX, x_is_f32, dy, n, c->d, c->dI8Scale, c->dI8Centre,
                                      c->dI8Flags, c->dI8NormSum, gate ? c->dI8NormSum + 1 : nullptr, c->stream));
    c->launches += 1;
    if (gate) {
      // AUTO's magnitude gate.  The distance contraction accumulates 2 x^.z^ - |x^|^2 - |z^|^2 in fp32 in tensor
      // memory; its rounding (toward zero, measured) scales with those magnitudes: at mean|x^|^2 + mean|z^|^2 ~ 4.4
      // the elements are good to 2.7e-7 rms (parity holds, tests), at ~12 (airfoil: norms up to 40) they are not
      // (posterior mean off by 5e-4).  Above the budget the shard goes to the fp64 DMMA kernel instead.
      double xsum = 0.0;
      SGP_CUDA(c, cudaMemcpyAsync(&xsum, c->dI8NormSum + 1, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
      SGP_CUDA(c, cudaStreamSynchronize(c->stream));
      if (xsum / static_cast<double>(n) + c->i8_z_norm_mean > c->i8_norm_budget) {
        // Large scaled norms mean tiny kernel values, and the fixed-point digits carry an ABSOLUTE error of 2^-24: on
        // such shards the int8 Gram -- with either distance form -- loses the posterior mean (airfoil-like data: 1.5e-4
        // to 1.5e-2 against 7e-7 .. 7e-6 of the fp64 kernel, profiles/r02o_i8_conditioning.txt).  fp64 DMMA kernel.
        use_i8 = false;
        path = 0;
      }
    }
  }
  I8Direct direct;
  if (path == 2) {
    const size_t xb = static_cast<size_t>((n + 63) / 64) * c->kf.n_terms * 64 * c->i8_dpad4 * sizeof(float);
    if (xb > c->i8_xt_bytes) {
      cudaFree(c->dI8Xt); c->dI8Xt = nullptr; c->i8_xt_bytes = 0;
      SGP_CUDA(c, cudaMalloc(&c->dI8Xt, xb));
      c->i8_xt_bytes = xb;
    }
    // AUTO applies the same magnitude budget as with tensor-core distances (on the WIDEST term's scaled squared norms: it
    // sets the size of the kernel values): first chunk here, whole window at finish
    rc = direct_prepare(c);
    if (rc != SGP_OK) return rc;
    const bool dgate = (c->precision == SGP_PREC_AUTO) && first_of_call;
    const bool dbudget = (c->precision == SGP_PREC_AUTO);
    if (dgate) SGP_CUDA(c, cudaMemsetAsync(c->dI8NormSum + 1, 0, sizeof(double), c->stream));
    SGP_CUDA(c, launch_i8_prep_points_direct(reinterpret_cast<float*>(c->dI8Xt), c->dI8Ys, dX, x_is_f32, dy, n, c->d,
                                             c->i8_dpad4, c->kf.n_terms, c->dI8DScale,
                                             c->dI8DScale + static_cast<size_t>(kMaxTerms) * c->i8_dpad4, c->dI8Flags,
                                             c->i8_direct_r2max, dbudget ? c->dI8NormSum : nullptr,
                                             dgate ? c->dI8NormSum + 1 : nullptr, c->stream));
    c->launches += 1;
    if (dgate) {
      double xsum = 0.0;
      SGP_CUDA(c, cudaMemcpyAsync(&xsum, c->dI8NormSum + 1, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
      SGP_CUDA(c, cudaStreamSynchronize(c->stream));
      if (xsum / static_cast<double>(n) + c->i8d_z_norm_mean > c->i8_norm_budget) path = 0;
    }
  }
  if (path == 2) {
    direct.on = 1; direct.n_terms = c->kf.n_terms; direct.dpad4 = c->i8_dpad4;
    double csum = 0.0;
    for (int t = 0; t < c->kf.n_terms; ++t) csum += c->kf.scale[t];
    for (int t = 0; t < c->kf.n_terms; ++t) direct.w[t] = static_cast<float>(c->kf.scale[t] / csum);
    direct.csum = csum;
    c->i8_direct_used = true;
  }
  if (first_of_call) c->call_path = path;
  if (use_i8 || path == 2) c->i8_points += n;
  if (use_i8) c->i8_used = true;
  c->last_path = (path == 1) ? SGP_PREC_I8 : (path == 2) ? SGP_PREC_I8_DIRECT
                 : (c->precision == SGP_PREC_F64_STRICT ? SGP_PREC_F64_STRICT : SGP_PREC_F64);
  if (c->gram_events_used == c->gram_events.size()) {          // grow the event pool (steady state: no creation)
    cudaEvent_t a, b;
    SGP_CUDA(c, cudaEventCreate(&a));
    SGP_CUDA(c, cudaEventCreate(&b));
    c->gram_events.emplace_back(a, b);
  }
  cudaEvent_t e0 = c->gram_events[c->gram_events_used].first, e1 = c->gram_events[c->gram_events_used].second;
  c->gram_events_used += 1;
  SGP_CUDA(c, cudaEventRecord(e0, c->stream));
  const size_t mm = static_cast<size_t>(c->m) * c->m;
  if (use_i8 && c->i8_impl == 0) {
    SGP_CUDA(c, launch_gram_i8(c->dI8Xt, c->dI8Ys, c->dI8Zt, n, c->d, c->m_pad, n_slices, c->dGpart, c->dBpart,
                               c->kf.scale[0], c->dbgT, c->dbgW, nullptr, c->stream));
    SGP_CUDA(c, cudaEventRecord(e1, c->stream));
    SGP_CUDA(c, launch_gram_reduce(c->dGb, c->dGb + mm, c->dGpart, c->dBpart, n_slices, c->m, c->m_pad, c->stream));
    c->launches += 2;
    return SGP_OK;
  }
  if (use_i8 || path == 2) {
    const uint8_t* zop = (path == 2) ? reinterpret_cast<const uint8_t*>(c->dI8Zd) : c->dI8Zt;
    for (int i = 0; i < n_plan; ++i) {
      SGP_CUDA(c, launch_gram_i8_ring(c->dI8Xt, c->dI8Ys, zop, n, c->d, c->m_pad, plan[i], direct, c->dGpart, c->dBpart,
                                 c->kf.scale[0], static_cast<uint8_t*>(c->i8_share.p), c->dbgT, c->dbgW, c->dbgClk,
                                 c->i8_pm_dev, c->stream));
      c->launches += 1;
    }
    SGP_CUDA(c, cudaEventRecord(e1, c->stream));
    for (int i = 0; i < n_plan; ++i) {          // deterministic slice reduction, per launch (its columns, its slices)
      SGP_CUDA(c, launch_gram_reduce_upper(c->dGb, c->dGb + mm, c->dGpart, c->dBpart, plan[i].n_slices, c->m, c->m_pad,
                                           plan[i].col_lo * kTile, plan[i].col_hi * kTile, c->stream));
      c->launches += 1;
    }
    return SGP_OK;
  }
  SGP_CUDA(c, launch_gram_f64(p, c->precision == SGP_PREC_F64_STRICT, c->stream));
  SGP_CUDA(c, cudaEventRecord(e1, c->stream));
  SGP_CUDA(c, launch_gram_reduce(c->dGb, c->dGb + mm, c->dGpart, c->dBpart, n_slices, c->m, c->m_pad, c->stream));
  c->launches += 2;
  return SGP_OK;
}

static void drop_gram_events(Ctx* c) {
  for (auto& e : c->gram_events) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
  c->gram_events.clear();
  c->gram_events_used = 0;
}

}  // namespace sgp

using namespace sgp;

extern "C" {

int sgp_version(void) { return 100; }

int sgp_ctx_create(sgp_ctx** out, int device) {
  if (!out) return fail(nullptr, SGP_E_BADARG, "out == NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, SGP_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                         " (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail(nullptr, SGP_E_BADARG, "device index out of range");
  Ctx* c = new (std::nothrow) Ctx();
  if (!c) return fail(nullptr, SGP_E_NOMEM, "out of host memory");
  c->device = device;
  auto bail = [&](int code, const std::string& m) { std::string mm = m; delete c; return fail(nullptr, code, mm); };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(SGP_E_CUDA, cudaGetErrorString(e));
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail(SGP_E_CUDA, cudaGetErrorString(e));
  if (prop.major != 10)
    return bail(SGP_E_CUDA, "this library is built for sm_100a (B200) only; device is sm_" +
                                std::to_string(prop.major) + std::to_string(prop.minor));
  c->num_sms = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)) != cudaSuccess)
    return bail(SGP_E_CUDA, cudaGetErrorString(e));
  for (int i = 0; i < 2; ++i) {
    cudaEventCreateWithFlags(&c->stage_free[i], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->stage_ready[i], cudaEventDisableTiming);
  }
  if ((e = cudaStreamCreateWithFlags(&c->tail_stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&c->tail_fork, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&c->tail_join, cudaEventDisableTiming)) != cudaSuccess)
    return bail(SGP_E_CUDA, cudaGetErrorString(e));
  if (cudaHostAlloc(reinterpret_cast<void**>(&c->i8_pm_host), 64, cudaHostAllocMapped) == cudaSuccess) {
    std::memset(c->i8_pm_host, 0, 64);
    if (cudaHostGetDevicePointer(&c->i8_pm_dev, c->i8_pm_host, 0) != cudaSuccess) c->i8_pm_dev = nullptr;
  }
  c->i8_impl = 1;                 // shared-panel ring kernel; SGP_I8_IMPL=v1 selects round 1's self-contained kernel
  if (const char* ev = getenv("SGP_I8_IMPL")) c->i8_impl = (std::string(ev) == "v1") ? 0 : 1;
  if (cusolverDnCreate(&c->solver) != CUSOLVER_STATUS_SUCCESS) return bail(SGP_E_CUDA, "cusolverDnCreate failed");
  if (cusolverDnCreate(&c->solver2) != CUSOLVER_STATUS_SUCCESS) return bail(SGP_E_CUDA, "cusolverDnCreate failed");
  if (cublasCreate(&c->blas) != CUBLAS_STATUS_SUCCESS) return bail(SGP_E_CUDA, "cublasCreate failed");
  *out = reinterpret_cast<sgp_ctx*>(c);
  return SGP_OK;
}

int sgp_ctx_destroy(sgp_ctx* h) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  drop_gram_events(c);
  for (auto& e : c->user_events) if (e) cudaEventDestroy(e);
  free_active_set(c);
  cudaFree(c->dGpart); cudaFree(c->dBpart);
  cudaFree(c->dEx); cudaFree(c->dEy); cudaFree(c->dEoff); cudaFree(c->dEf); cudaFree(c->dNllPer); cudaFree(c->dNllScratch);
  cudaFree(c->dI8Xt); cudaFree(c->dI8Ys); cudaFree(c->dbgT); cudaFree(c->dbgW); cudaFree(c->dbgClk); cudaFree(c->i8_share.p);
  for (int i = 0; i < 2; ++i) {
    cudaFree(c->stageX[i]); cudaFree(c->stageY[i]);
    if (c->stage_free[i]) cudaEventDestroy(c->stage_free[i]);
    if (c->stage_ready[i]) cudaEventDestroy(c->stage_ready[i]);
  }
  if (c->comm && nccl().ok) nccl().CommDestroy(c->comm);
  if (c->i8_pm_host) cudaFreeHost(c->i8_pm_host);
  cudaFree(c->greedy_ws.p); cudaFree(c->sweep_ws.p); cudaFree(c->bcm_ws.p); cudaFree(c->tail_ws.p); cudaFree(c->tail_ws2.p); cudaFree(c->predict_ws.p); cudaFree(c->cross_ws.p);
  if (c->tail_fork) cudaEventDestroy(c->tail_fork);
  if (c->tail_join) cudaEventDestroy(c->tail_join);
  if (c->tail_stream) cudaStreamDestroy(c->tail_stream);
  if (c->solver) cusolverDnDestroy(c->solver);
  if (c->solver2) cusolverDnDestroy(c->solver2);
  if (c->blas) cublasDestroy(c->blas);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  delete c;
  return SGP_OK;
}

const char* sgp_last_error(const sgp_ctx* h) {
  const Ctx* c = reinterpret_cast<const Ctx*>(h);
  return c ? c->err.c_str() : g_create_err.c_str();
}

int sgp_set_precision(sgp_ctx* h, int mode) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (mode < SGP_PREC_F64 || mode > SGP_PREC_I8_DIRECT) return fail(c, SGP_E_BADARG, "unknown precision mode");
  c->precision = mode;
  return SGP_OK;
}

int sgp_comm_unique_id(void* out128) {
  if (!out128) return SGP_E_BADARG;
  static_assert(sizeof(ncclUniqueId) <= SGP_UNIQUE_ID_BYTES, "ncclUniqueId does not fit");
  if (!nccl().ok) return fail(nullptr, SGP_E_NCCL, "libnccl.so.2 could not be loaded");
  ncclUniqueId id;
  if (nccl().GetUniqueId(&id) != ncclSuccess) return fail(nullptr, SGP_E_NCCL, "ncclGetUniqueId failed");
  std::memset(out128, 0, SGP_UNIQUE_ID_BYTES);
  std::memcpy(out128, &id, sizeof(id));
  return SGP_OK;
}

int sgp_comm_init(sgp_ctx* h, const void* id128, int rank, int nranks) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(c, SGP_E_BADARG, "bad comm arguments");
  if (!nccl().ok) return fail(c, SGP_E_NCCL, "libnccl.so.2 could not be loaded");
  SGP_CUDA(c, cudaSetDevice(c->device));
  ncclUniqueId id;
  std::memcpy(&id, id128, sizeof(id));
  ncclResult_t r = nccl().CommInitRank(&c->comm, nranks, id, rank);
  if (r != ncclSuccess) return fail(c, SGP_E_NCCL, std::string("ncclCommInitRank: ") + nccl().GetErrorString(r));
  c->rank = rank; c->nranks = nranks;
  return SGP_OK;
}

int sgp_stats_begin(sgp_ctx* h, const sgp_kernel_desc* k, const double* Z, int32_t m, int32_t d) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!k || !Z || m <= 0 || d <= 0 || k->n_terms <= 0 || !k->terms)
    return fail(c, SGP_E_BADARG, "sgp_stats_begin: null or empty argument");
  SGP_CUDA(c, cudaSetDevice(c->device));
  // ---- flatten: drop Eye terms from the cross path (kernel/Kernel.scala:157), sum their coefficients ----
  KernelFlat kf;
  const int dpad = (d + 3) & ~3;
  std::vector<double> beta(static_cast<size_t>(kMaxTerms) * dpad, 0.0);
  for (int t = 0; t < k->n_terms; ++t) {
    const sgp_kernel_term& term = k->terms[t];
    if (!(term.scale >= 0.0)) return fail(c, SGP_E_BADARG, "requirement failed: C should be positive");
    kf.self_kernel += term.scale;
    if (term.type == SGP_TERM_EYE) { kf.eye_sum += term.scale; continue; }
    if (kf.n_terms == kMaxTerms) return fail(c, SGP_E_BADARG, "too many non-Eye kernel terms (max 4)");
    double* bt = beta.data() + static_cast<size_t>(kf.n_terms) * dpad;
    if (term.type == SGP_TERM_ARD) {
      if (!term.beta) return fail(c, SGP_E_BADARG, "ARD term without beta");
      for (int j = 0; j < d; ++j) bt[j] = term.beta[j];
    } else if (term.type == SGP_TERM_RBF) {
      if (!(term.sigma > 0.0)) return fail(c, SGP_E_BADARG, "RBF sigma must be > 0");
      // exp(-|x-z|^2 / (2 sigma^2)) = exp(-sum_k (x_k - z_k)^2 beta^2), beta = 1/(sqrt(2) sigma)
      for (int j = 0; j < d; ++j) bt[j] = 1.0 / (std::sqrt(2.0) * term.sigma);
    } else {
      return fail(c, SGP_E_BADARG, "unknown kernel term type");
    }
    kf.scale[kf.n_terms++] = term.scale;
  }
  // device buffers are kept across begin() calls with the same (m, d, term count): cudaMalloc/cudaFree are
  // synchronising and cost milliseconds -- more than the whole statistics pass on a B200
  const int nt = kf.n_terms > 0 ? kf.n_terms : 1;
  const bool same_shape = c->dZ && c->m == m && c->d == d && c->alloc_terms == nt;
  if (!same_shape) {
    SGP_CUDA(c, cudaStreamSynchronize(c->stream));
    free_active_set(c);
  }
  c->m = m; c->d = d; c->dpad = dpad; c->m_pad = (m + kTile - 1) / kTile * kTile; c->kf = kf;
  const size_t mm = static_cast<size_t>(m) * m;
  if (!same_shape) {
    c->alloc_terms = nt;
    SGP_CUDA(c, cudaMalloc(&c->dZ, static_cast<size_t>(m) * d * 8));
    SGP_CUDA(c, cudaMalloc(&c->dZs, static_cast<size_t>(nt) * c->m_pad * dpad * 8));
    SGP_CUDA(c, cudaMalloc(&c->dBeta, static_cast<size_t>(kMaxTerms) * dpad * 8));
    SGP_CUDA(c, cudaMalloc(&c->dGb, (mm + m + 1) * 8));     // [G ; b ; status] -- one all-reduce
    SGP_CUDA(c, cudaMalloc(&c->dMagicVec, static_cast<size_t>(m) * 8));
    SGP_CUDA(c, cudaMalloc(&c->dMagicMat, mm * 8));
  }
  SGP_CUDA(c, cudaMemcpyAsync(c->dZ, Z, static_cast<size_t>(m) * d * 8, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaMemcpyAsync(c->dBeta, beta.data(), beta.size() * 8, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaMemsetAsync(c->dGb, 0, (mm + m + 1) * 8, c->stream));
  for (int t = 0; t < kf.n_terms; ++t) {
    SGP_CUDA(c, launch_scale_rows(c->dZs + static_cast<size_t>(t) * c->m_pad * dpad, c->dZ,
                                  c->dBeta + static_cast<size_t>(t) * dpad, m, c->m_pad, d, dpad, c->stream));
    c->launches += 1;
  }
  // ---- tcgen05 int8 path: qualifies for one non-Eye term and d <= 32 (two 64-column K chunks) -------------
  c->i8_ok = (kf.n_terms == 1 && d <= 32);
  std::vector<double> sc16, ctr16;               // live until the synchronisation at the end of this function
  if (!c->dI8Flags) {
    SGP_CUDA(c, cudaMalloc(&c->dI8Flags, sizeof(int)));
    SGP_CUDA(c, cudaMalloc(&c->dI8NormSum, 2 * sizeof(double)));
  }
  SGP_CUDA(c, cudaMemsetAsync(c->dI8Flags, 0, sizeof(int), c->stream));
  SGP_CUDA(c, cudaMemsetAsync(c->dI8NormSum, 0, 2 * sizeof(double), c->stream));
  if (c->i8_ok) {
    const int dp16 = (d + 15) / 16 * 16;
    std::vector<double>& sc = sc16; std::vector<double>& ctr = ctr16;
    sc.assign(dp16, 0.0); ctr.assign(dp16, 0.0);
    const double s2 = std::sqrt(1.4426950408889634074);          // sqrt(log2 e): exponent in base 2
    for (int j = 0; j < d; ++j) {
      sc[j] = s2 * beta[j];
      double acc = 0.0;
      for (int i = 0; i < m; ++i) acc += Z[static_cast<size_t>(i) * d + j];
      ctr[j] = acc / m;                                          // distances are translation invariant
    }
    if (!c->dI8Scale) {
      SGP_CUDA(c, cudaMalloc(&c->dI8Scale, dp16 * 8));
      SGP_CUDA(c, cudaMalloc(&c->dI8Centre, dp16 * 8));
      SGP_CUDA(c, cudaMalloc(&c->dI8Zt, i8_active_scratch_bytes(c->m_pad, i8_nchunks(d))));
    }
    {
      double zsum = 0.0;
      for (int i = 0; i < m; ++i)
        for (int j = 0; j < d; ++j) {
          const double v = (Z[static_cast<size_t>(i) * d + j] - ctr[j]) * sc[j];
          zsum += v * v;
        }
      c->i8_z_norm_mean = zsum / m;
      if (const char* e = getenv("SGP_I8_NORM_BUDGET")) c->i8_norm_budget = atof(e);
    }
    SGP_CUDA(c, cudaMemcpyAsync(c->dI8Scale, sc.data(), dp16 * 8, cudaMemcpyHostToDevice, c->stream));
    SGP_CUDA(c, cudaMemcpyAsync(c->dI8Centre, ctr.data(), dp16 * 8, cudaMemcpyHostToDevice, c->stream));
    SGP_CUDA(c, launch_i8_prep_active(c->dI8Zt, c->dZ, m, c->m_pad, d, c->dI8Scale, c->dI8Centre, c->dI8Flags,
                                      c->stream));
    c->launches += 1;
  }
  // ---- direct-distance mode of the int8 Gram: 1..4 non-Eye terms, n_terms * dpad4 <= 72 (smem) ------------
  {
    const int dpad4 = (d + 3) & ~3;
    c->i8_direct_ok = kf.n_terms >= 1 && kf.n_terms * dpad4 <= 72;
    if (c->i8_direct_ok) {
      c->i8_dpad4 = dpad4;
      if (const char* e = getenv("SGP_I8_DIRECT_R2MAX")) c->i8_direct_r2max = static_cast<float>(atof(e));
      std::vector<double>& sc = c->i8d_sc;                                           // [term][k] scales, then the centre
      sc.assign(static_cast<size_t>(kMaxTerms + 1) * dpad4, 0.0);
      const double s2 = std::sqrt(1.4426950408889634074);
      for (int t = 0; t < kf.n_terms; ++t)
        for (int j = 0; j < d; ++j) sc[static_cast<size_t>(t) * dpad4 + j] = s2 * beta[static_cast<size_t>(t) * dpad + j];
      for (int j = 0; j < d; ++j) {
        double acc = 0.0;
        for (int i = 0; i < m; ++i) acc += Z[static_cast<size_t>(i) * d + j];
        sc[static_cast<size_t>(kMaxTerms) * dpad4 + j] = acc / m;
      }
      {                                                   // mean scaled squared norm of the active set, widest term
        double best = 1e300;
        for (int t = 0; t < kf.n_terms; ++t) {
          double zsum = 0.0;
          for (int i = 0; i < m; ++i)
            for (int j = 0; j < d; ++j) {
              const double v = (Z[static_cast<size_t>(i) * d + j] - sc[static_cast<size_t>(kMaxTerms) * dpad4 + j]) *
                               sc[static_cast<size_t>(t) * dpad4 + j];
              zsum += v * v;
            }
          best = std::min(best, zsum / m);
        }
        c->i8d_z_norm_mean = best;
        if (const char* e = getenv("SGP_I8_NORM_BUDGET")) c->i8_norm_budget = atof(e);
      }
      // the device side (scales upload, active-set tiles) is prepared on first use of the mode: direct_prepare()
    }
  }
  c->i8d_prepared = false;
  c->i8_direct_used = false;
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));   // Z / beta are host temporaries of the caller
  c->gram_events_used = 0;
  c->i8_points = 0;
  c->begun = true; c->finished = false; c->has_magic = false; c->i8_used = false;
  return SGP_OK;
}

int sgp_stats_accumulate_device(sgp_ctx* h, const void* dX, int32_t x_is_f32, const double* dy, int64_t n) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->begun || c->finished) return fail(c, SGP_E_STATE, "sgp_stats_begin should have been called first");
  if (n < 0 || (n > 0 && (!dX || !dy))) return fail(c, SGP_E_BADARG, "null shard");
  SGP_CUDA(c, cudaSetDevice(c->device));
  if (c->kf.n_terms == 0) return SGP_OK;   // only Eye terms: the cross kernel is identically zero
  return launch_stats(c, dX, x_is_f32, dy, n, n, true);
}

int sgp_stats_accumulate(sgp_ctx* h, const void* X, int32_t x_is_f32, const double* y, int64_t n) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->begun || c->finished) return fail(c, SGP_E_STATE, "sgp_stats_begin should have been called first");
  if (n < 0 || (n > 0 && (!X || !y))) return fail(c, SGP_E_BADARG, "null shard");
  if (n == 0 || c->kf.n_terms == 0) return SGP_OK;
  SGP_CUDA(c, cudaSetDevice(c->device));
  const size_t esz = x_is_f32 ? 4 : 8;
  const size_t row = static_cast<size_t>(c->d) * esz;
  // chunk so that copy (PCIe) and compute overlap: ~16 MB of X per chunk (the first chunk's copy is the exposed part:
  // 0.3 ms at 55 GB/s), at least 64k points
  long long chunk = static_cast<long long>((16u << 20) / row);
  if (chunk < 65536) chunk = 65536;
  {                                           // equal chunks (multiples of 64 points) instead of a short tail chunk
    const long long nchunks = (n + chunk - 1) / chunk;
    chunk = ((n + nchunks - 1) / nchunks + 63) / 64 * 64;
  }
  if (chunk > n) chunk = n;
  // The first chunk's copy is the only one the kernels cannot hide: make it a quarter of the others
  long long first = chunk;
  if (n > chunk) {
    first = (chunk / 4 + 63) / 64 * 64;
    if (first < 65536) first = 65536;
    if (first > chunk) first = chunk;
    const long long rest = n - first;
    const long long nchunks = (rest + chunk - 1) / chunk;
    chunk = ((rest + nchunks - 1) / nchunks + 63) / 64 * 64;
    if (chunk < first) chunk = first;
  }
  if (chunk > c->stage_points || row * chunk > c->stage_bytes) {
    SGP_CUDA(c, cudaStreamSynchronize(c->stream));
    SGP_CUDA(c, cudaStreamSynchronize(c->copy_stream));
    for (int i = 0; i < 2; ++i) {
      cudaFree(c->stageX[i]); cudaFree(c->stageY[i]);
      c->stageX[i] = nullptr; c->stageY[i] = nullptr;
      SGP_CUDA(c, cudaMalloc(&c->stageX[i], row * chunk));
      SGP_CUDA(c, cudaMalloc(&c->stageY[i], static_cast<size_t>(chunk) * 8));
      SGP_CUDA(c, cudaEventRecord(c->stage_free[i], c->stream));
    }
    c->stage_bytes = row * chunk; c->stage_points = chunk;
  }
  const char* Xb = static_cast<const char*>(X);
  int buf = 0;
  for (long long p0 = 0, step = first; p0 < n; p0 += step, step = chunk, buf ^= 1) {
    const long long cn = (n - p0 < step) ? (n - p0) : step;
    SGP_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->stage_free[buf], 0));
    SGP_CUDA(c, cudaMemcpyAsync(c->stageX[buf], Xb + static_cast<size_t>(p0) * row, row * cn, cudaMemcpyHostToDevice,
                                c->copy_stream));
    SGP_CUDA(c, cudaMemcpyAsync(c->stageY[buf], y + p0, static_cast<size_t>(cn) * 8, cudaMemcpyHostToDevice,
                                c->copy_stream));
    SGP_CUDA(c, cudaEventRecord(c->stage_ready[buf], c->copy_stream));
    SGP_CUDA(c, cudaStreamWaitEvent(c->stream, c->stage_ready[buf], 0));
    int rc = launch_stats(c, c->stageX[buf], x_is_f32, c->stageY[buf], cn, n, p0 == 0);
    if (rc != SGP_OK) return rc;
    SGP_CUDA(c, cudaEventRecord(c->stage_free[buf], c->stream));
  }
  // the caller may reuse / free X, y as soon as we return
  SGP_CUDA(c, cudaStreamSynchronize(c->copy_stream));
  return SGP_OK;
}

int sgp_stats_finish(sgp_ctx* h, double* G_out, double* b_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->begun) return fail(c, SGP_E_STATE, "sgp_stats_begin should have been called first");
  SGP_CUDA(c, cudaSetDevice(c->device));
  const size_t mm = static_cast<size_t>(c->m) * c->m;
  double status = 0.0;
  if (!c->finished) {
    // The rank-local status of the int8 path (fp16 operand range overflow; AUTO's magnitude budget exceeded over the
    // WHOLE window, not just the first chunk the kernel choice looked at) rides in the last slot of the all-reduced
    // buffer: every rank sees the same sum and takes the same return decision AFTER the collective -- a rank that
    // bailed out before it would leave its peers blocked in ncclAllReduce.
    const bool i8 = c->i8_ok && c->i8_used && c->dI8Flags;
    const bool i8d = c->i8_direct_used && c->dI8Flags;          // direct mode: bit 2 = scaled squared norm above its limit
    const bool budget = (i8 || i8d) && c->precision == SGP_PREC_AUTO;
    const double zmean = (i8 && i8d) ? std::min(c->i8_z_norm_mean, c->i8d_z_norm_mean) : (i8 ? c->i8_z_norm_mean : c->i8d_z_norm_mean);
    const double limit = (c->i8_norm_budget - zmean) * static_cast<double>(c->i8_points) * 1.25;
    SGP_CUDA(c, launch_status_to_double(c->dGb + mm + c->m, (i8 || i8d) ? c->dI8Flags : nullptr, (i8 ? 1 : 0) | (i8d ? 4 : 0),
                                        budget ? c->dI8NormSum : nullptr, limit, c->stream));
    c->launches += 1;
    if (c->comm && c->nranks > 1) {
      // PGPH:31-35 combOp: one all-reduce of the packed [G;b;status] over NVLink
      ncclResult_t r = nccl().AllReduce(c->dGb, c->dGb, mm + c->m + 1, ncclDouble, ncclSum, c->comm, c->stream);
      if (r != ncclSuccess) return fail(c, SGP_E_NCCL, std::string("ncclAllReduce: ") + nccl().GetErrorString(r));
      c->launches += 1;
    }
    SGP_CUDA(c, cudaMemcpyAsync(&status, c->dGb + mm + c->m, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  }
  c->finished = true;
  if (G_out) SGP_CUDA(c, cudaMemcpyAsync(G_out, c->dGb, mm * 8, cudaMemcpyDeviceToHost, c->stream));
  if (b_out)
    SGP_CUDA(c, cudaMemcpyAsync(b_out, c->dGb + mm, static_cast<size_t>(c->m) * 8, cudaMemcpyDeviceToHost, c->stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  if (status != 0.0)
    return fail(c, SGP_E_RANGE, "the int8 path cannot represent this shard on some rank (scaled coordinates outside the "
                                "fp16 operand range, scaled squared norms above AUTO's magnitude budget for tensor-core "
                                "distances, or above the fp32 direct-distance limit); rerun the statistics with "
                                "sgp_set_precision(SGP_PREC_I8_DIRECT) or sgp_set_precision(SGP_PREC_F64)");
  return SGP_OK;
}

int sgp_sync(sgp_ctx* h) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  SGP_CUDA(c, cudaSetDevice(c->device));
  SGP_CUDA(c, cudaStreamSynchronize(c->copy_stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  return SGP_OK;
}

int sgp_magic(sgp_ctx* h, const double* G_in, const double* b_in, double* magic_vector, double* magic_matrix) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->begun) return fail(c, SGP_E_STATE, "sgp_stats_begin should have been called first");
  if ((G_in == nullptr) != (b_in == nullptr)) return fail(c, SGP_E_BADARG, "G_in and b_in must be given together");
  SGP_CUDA(c, cudaSetDevice(c->device));
  const size_t mm = static_cast<size_t>(c->m) * c->m;
  if (G_in) {
    SGP_CUDA(c, cudaMemcpyAsync(c->dGb, G_in, mm * 8, cudaMemcpyHostToDevice, c->stream));
    SGP_CUDA(c, cudaMemcpyAsync(c->dGb + mm, b_in, static_cast<size_t>(c->m) * 8, cudaMemcpyHostToDevice, c->stream));
    c->finished = true;
  } else if (!c->finished) {
    return fail(c, SGP_E_STATE, "sgp_stats_finish should have been called first");
  }
  return run_tail(c, magic_vector, magic_matrix);
}

int sgp_set_magic(sgp_ctx* h, const double* v, const double* M) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->begun) return fail(c, SGP_E_STATE, "sgp_stats_begin should have been called first");
  if (!v || !M) return fail(c, SGP_E_BADARG, "sgp_set_magic: null argument");
  SGP_CUDA(c, cudaSetDevice(c->device));
  const size_t mm = static_cast<size_t>(c->m) * c->m;
  SGP_CUDA(c, cudaMemcpyAsync(c->dMagicVec, v, static_cast<size_t>(c->m) * 8, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaMemcpyAsync(c->dMagicMat, M, mm * 8, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));          // the caller may reuse v, M as soon as we return
  c->has_magic = true;
  return SGP_OK;
}

int sgp_predict(sgp_ctx* h, const double* X, int64_t n, double* mean_out, double* var_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->has_magic) return fail(c, SGP_E_STATE, "sgp_magic should have been called first");
  if (n < 0 || (n > 0 && (!X || !mean_out))) return fail(c, SGP_E_BADARG, "null argument");
  if (n == 0) return SGP_OK;
  SGP_CUDA(c, cudaSetDevice(c->device));
  return run_predict(c, X, n, mean_out, var_out);
}

int64_t sgp_launch_count(const sgp_ctx* h) {
  const Ctx* c = reinterpret_cast<const Ctx*>(h);
  return c ? c->launches : 0;
}

int sgp_gram_kernel_time(sgp_ctx* h, double* total_ms, int64_t* launches) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  SGP_CUDA(c, cudaSetDevice(c->device));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  double tot = 0.0;
  for (size_t i = 0; i < c->gram_events_used; ++i) {
    float ms = 0.f;
    SGP_CUDA(c, cudaEventElapsedTime(&ms, c->gram_events[i].first, c->gram_events[i].second));
    tot += ms;
  }
  if (total_ms) *total_ms = tot;
  if (launches) *launches = static_cast<int64_t>(c->gram_events_used);
  return SGP_OK;
}

int sgp_experts_upload(sgp_ctx* h, const double* X, const double* y, const int64_t* offsets, int64_t E, int32_t d) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!X || !y || !offsets || E <= 0 || d <= 0) return fail(c, SGP_E_BADARG, "sgp_experts_upload: null or empty argument");
  SGP_CUDA(c, cudaSetDevice(c->device));
  const long long n = offsets[E];
  int nmax = 0;
  for (int64_t e = 0; e < E; ++e) {
    const long long ne = offsets[e + 1] - offsets[e];
    if (ne <= 0) return fail(c, SGP_E_BADARG, "empty expert");
    if (ne > nmax) nmax = static_cast<int>(ne);
  }
  // (no upper bound on the expert size -- GaussianProcessParams.scala:36: experts above the on-chip kernel's 168 points
  //  take the global-memory LU path of sgp_bcm_nll)
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaFree(c->dEx); cudaFree(c->dEy); cudaFree(c->dEoff); cudaFree(c->dEf);
  c->dEx = c->dEy = c->dEf = nullptr; c->dEoff = nullptr;
  SGP_CUDA(c, cudaMalloc(&c->dEx, static_cast<size_t>(n) * d * 8));
  SGP_CUDA(c, cudaMalloc(&c->dEy, static_cast<size_t>(n) * 8));
  SGP_CUDA(c, cudaMalloc(&c->dEoff, static_cast<size_t>(E + 1) * 8));
  SGP_CUDA(c, cudaMalloc(&c->dEf, static_cast<size_t>(n) * 8));
  SGP_CUDA(c, cudaMemsetAsync(c->dEf, 0, static_cast<size_t>(n) * 8, c->stream));   // f = zeros (GPCls:54)
  SGP_CUDA(c, cudaMemcpyAsync(c->dEx, X, static_cast<size_t>(n) * d * 8, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaMemcpyAsync(c->dEy, y, static_cast<size_t>(n) * 8, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaMemcpyAsync(c->dEoff, offsets, static_cast<size_t>(E + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  c->n_experts = E; c->ex_d = d; c->ex_nmax = nmax; c->ex_n = n;
  return SGP_OK;
}

int sgp_experts_upload_grouped(sgp_ctx* h, const void* X, int32_t x_is_f32, const double* y, int64_t n, int32_t d,
                               int32_t dataset_size_for_expert) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!X || !y || n <= 0 || d <= 0 || dataset_size_for_expert <= 0)
    return fail(c, SGP_E_BADARG, "sgp_experts_upload_grouped: null or empty argument");
  SGP_CUDA(c, cudaSetDevice(c->device));
  // GPC:27  numberOfExperts = Math.round(points.count() / datasetSizeForExpert)  (round half up on a positive double)
  const long long E = static_cast<long long>(std::floor(static_cast<double>(n) / dataset_size_for_expert + 0.5));
  if (E <= 0) return fail(c, SGP_E_BADARG, "numberOfExperts == 0 (N < datasetSizeForExpert / 2): the reference fails with / by zero");
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaFree(c->dEx); cudaFree(c->dEy); cudaFree(c->dEoff); cudaFree(c->dEf);
  c->dEx = c->dEy = c->dEf = nullptr; c->dEoff = nullptr;
  SGP_CUDA(c, cudaMalloc(&c->dEx, static_cast<size_t>(n) * d * 8));
  SGP_CUDA(c, cudaMalloc(&c->dEy, static_cast<size_t>(n) * 8));
  SGP_CUDA(c, cudaMalloc(&c->dEoff, static_cast<size_t>(E + 1) * 8));
  SGP_CUDA(c, cudaMalloc(&c->dEf, static_cast<size_t>(n) * 8));
  SGP_CUDA(c, cudaMemsetAsync(c->dEf, 0, static_cast<size_t>(n) * 8, c->stream));   // f = zeros (GPCls:54)
  SGP_CUDA(c, launch_expert_offsets(c->dEoff, n, E, c->stream));
  // stream the row-major input through the double-buffered staging area of the statistics path, gather on the device
  const size_t esz = x_is_f32 ? 4 : 8;
  const size_t row = static_cast<size_t>(d) * esz;
  long long chunk = static_cast<long long>((32u << 20) / row);
  if (chunk < 65536) chunk = 65536;
  if (chunk > n) chunk = n;
  if (chunk > c->stage_points || row * chunk > c->stage_bytes) {
    SGP_CUDA(c, cudaStreamSynchronize(c->copy_stream));
    for (int i = 0; i < 2; ++i) {
      cudaFree(c->stageX[i]); cudaFree(c->stageY[i]);
      c->stageX[i] = nullptr; c->stageY[i] = nullptr;
      SGP_CUDA(c, cudaMalloc(&c->stageX[i], row * chunk));
      SGP_CUDA(c, cudaMalloc(&c->stageY[i], static_cast<size_t>(chunk) * 8));
      SGP_CUDA(c, cudaEventRecord(c->stage_free[i], c->stream));
    }
    c->stage_bytes = row * chunk; c->stage_points = chunk;
  }
  const char* Xb = static_cast<const char*>(X);
  int buf = 0;
  for (long long p0 = 0; p0 < n; p0 += chunk, buf ^= 1) {
    const long long cn = (n - p0 < chunk) ? (n - p0) : chunk;
    SGP_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->stage_free[buf], 0));
    SGP_CUDA(c, cudaMemcpyAsync(c->stageX[buf], Xb + static_cast<size_t>(p0) * row, row * cn, cudaMemcpyHostToDevice, c->copy_stream));
    SGP_CUDA(c, cudaMemcpyAsync(c->stageY[buf], y + p0, static_cast<size_t>(cn) * 8, cudaMemcpyHostToDevice, c->copy_stream));
    SGP_CUDA(c, cudaEventRecord(c->stage_ready[buf], c->copy_stream));
    SGP_CUDA(c, cudaStreamWaitEvent(c->stream, c->stage_ready[buf], 0));
    SGP_CUDA(c, launch_group_experts(c->dEx, c->dEy, c->stageX[buf], x_is_f32, c->stageY[buf], n, d, E, p0, cn, c->stream));
    SGP_CUDA(c, cudaEventRecord(c->stage_free[buf], c->stream));
    c->launches += 1;
  }
  SGP_CUDA(c, cudaStreamSynchronize(c->copy_stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  const long long kq = n / E;
  c->n_experts = E; c->ex_d = d; c->ex_nmax = static_cast<int>(kq + ((n % E) ? 1 : 0)); c->ex_n = n;
  return SGP_OK;
}

namespace {
struct ObjectiveArgs {          // device-side view of (kernel, hyper-parameter descriptors) for the per-expert objectives
  KernelFlat kf;
  int W = 0;                    // 1 + n_hypers
  int any_ard = 0;              // some hyper-parameter is an ARD beta (per-dimension sums needed)
  double *dBeta = nullptr, *dCoef = nullptr, *dValue = nullptr, *dTotal = nullptr;
  int *dKind = nullptr, *dTerm = nullptr, *dDim = nullptr, *dFlags = nullptr;
};

// Flattens the kernel (same rules as sgp_stats_begin: Eye terms only add to the diagonal), maps the hyper-parameter
// descriptors onto the flattened terms and uploads everything into one scratch allocation.
int objective_setup(Ctx* c, const sgp_kernel_desc* k, const sgp_hyper* hypers, int nh, ObjectiveArgs& o) {
  if (!c->dEx) return fail(c, SGP_E_STATE, "sgp_experts_upload should have been called first");
  if (!k || !k->terms || k->n_terms <= 0 || nh < 0 || (nh > 0 && !hypers)) return fail(c, SGP_E_BADARG, "null argument");
  if (nh > bcm_nll_max_hypers()) return fail(c, SGP_E_BADARG, "too many hyper-parameters");
  const int d = c->ex_d;
  KernelFlat kf;
  std::vector<int> flat_of(k->n_terms, -1);
  std::vector<double> beta(static_cast<size_t>(kMaxTerms) * d, 0.0);
  for (int t = 0; t < k->n_terms; ++t) {
    const sgp_kernel_term& term = k->terms[t];
    if (!(term.scale >= 0.0)) return fail(c, SGP_E_BADARG, "requirement failed: C should be positive");
    if (term.type == SGP_TERM_EYE) { kf.eye_sum += term.scale; continue; }
    if (kf.n_terms == kMaxTerms) return fail(c, SGP_E_BADARG, "too many non-Eye kernel terms (max 4)");
    double* bt = beta.data() + static_cast<size_t>(kf.n_terms) * d;
    if (term.type == SGP_TERM_ARD) {
      if (!term.beta) return fail(c, SGP_E_BADARG, "ARD term without beta");
      for (int j = 0; j < d; ++j) bt[j] = term.beta[j];
    } else if (term.type == SGP_TERM_RBF) {
      if (!(term.sigma > 0.0)) return fail(c, SGP_E_BADARG, "RBF sigma must be > 0");
      for (int j = 0; j < d; ++j) bt[j] = 1.0 / (std::sqrt(2.0) * term.sigma);
    } else {
      return fail(c, SGP_E_BADARG, "unknown kernel term type");
    }
    flat_of[t] = kf.n_terms;
    kf.scale[kf.n_terms++] = term.scale;
  }
  const int W = 1 + nh;
  std::vector<int> kind(nh), hterm(nh, 0), hdim(nh, 0);
  std::vector<double> coef(static_cast<size_t>(nh) * (kMaxTerms + 1), 0.0), value(nh, 0.0);
  for (int i = 0; i < nh; ++i) {
    kind[i] = hypers[i].kind;
    value[i] = hypers[i].value;
    if (hypers[i].kind == SGP_HYPER_SCALE) {
      if (!hypers[i].coef) return fail(c, SGP_E_BADARG, "SCALE hyper-parameter without coef");
      for (int t = 0; t < k->n_terms; ++t) {
        const size_t col = (flat_of[t] >= 0) ? static_cast<size_t>(flat_of[t]) : static_cast<size_t>(kMaxTerms);
        coef[static_cast<size_t>(i) * (kMaxTerms + 1) + col] += hypers[i].coef[t];
      }
    } else if (hypers[i].kind == SGP_HYPER_ARD_BETA || hypers[i].kind == SGP_HYPER_RBF_SIGMA) {
      if (hypers[i].term < 0 || hypers[i].term >= k->n_terms || flat_of[hypers[i].term] < 0)
        return fail(c, SGP_E_BADARG, "hyper-parameter refers to a bad term");
      hterm[i] = flat_of[hypers[i].term];
      hdim[i] = hypers[i].dim;
      if (hypers[i].kind == SGP_HYPER_ARD_BETA) o.any_ard = 1;
      if (hypers[i].kind == SGP_HYPER_ARD_BETA && (hdim[i] < 0 || hdim[i] >= d)) return fail(c, SGP_E_BADARG, "bad ARD dim");
    } else {
      return fail(c, SGP_E_BADARG, "unknown hyper-parameter kind");
    }
  }
  // one scratch allocation: [beta | coef | value | total] doubles, then [kind | term | dim | flags] ints
  const size_t n_dbl = beta.size() + coef.size() + value.size() + W + 1;    // ... + totals [W] + status [1]
  const size_t n_int = 3 * static_cast<size_t>(nh) + 1;
  std::vector<double> hd(n_dbl, 0.0);
  std::vector<int> hi(n_int, 0);
  std::copy(beta.begin(), beta.end(), hd.begin());
  std::copy(coef.begin(), coef.end(), hd.begin() + beta.size());
  std::copy(value.begin(), value.end(), hd.begin() + beta.size() + coef.size());
  std::copy(kind.begin(), kind.end(), hi.begin());
  std::copy(hterm.begin(), hterm.end(), hi.begin() + nh);
  std::copy(hdim.begin(), hdim.end(), hi.begin() + 2 * nh);
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaFree(c->dNllScratch); c->dNllScratch = nullptr;
  SGP_CUDA(c, cudaMalloc(&c->dNllScratch, n_dbl * 8 + n_int * 4));
  double* dD = static_cast<double*>(c->dNllScratch);
  int* dI = reinterpret_cast<int*>(dD + n_dbl);
  SGP_CUDA(c, cudaMemcpyAsync(dD, hd.data(), n_dbl * 8, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaMemcpyAsync(dI, hi.data(), n_int * 4, cudaMemcpyHostToDevice, c->stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));          // hd / hi are locals
  const size_t per_bytes = static_cast<size_t>(c->n_experts) * W * 8;
  if (per_bytes > c->nll_per_cap) {
    cudaFree(c->dNllPer); c->dNllPer = nullptr; c->nll_per_cap = 0;
    SGP_CUDA(c, cudaMalloc(&c->dNllPer, per_bytes));
    c->nll_per_cap = per_bytes;
  }
  o.kf = kf; o.W = W;
  o.dBeta = dD; o.dCoef = dD + beta.size(); o.dValue = o.dCoef + coef.size(); o.dTotal = o.dValue + value.size();
  o.dKind = dI; o.dTerm = dI + nh; o.dDim = dI + 2 * nh; o.dFlags = dI + 3 * nh;
  return SGP_OK;
}

// all-reduce over ranks, copy the (objective, gradient) row back, map a bad pivot to SGP_E_NOT_PD
int objective_finish(Ctx* c, const ObjectiveArgs& o, double* val_out, double* grad_out, int mask, int err_code,
                     const char* err_msg) {
  // the rank-local status flag is all-reduced WITH the totals so that every rank raises (or none does)
  SGP_CUDA(c, launch_status_to_double(o.dTotal + o.W, o.dFlags, mask, nullptr, 0.0, c->stream));
  c->launches += 1;
  if (c->comm && c->nranks > 1) {
    ncclResult_t r = nccl().AllReduce(o.dTotal, o.dTotal, o.W + 1, ncclDouble, ncclSum, c->comm, c->stream);
    if (r != ncclSuccess) return fail(c, SGP_E_NCCL, std::string("ncclAllReduce: ") + nccl().GetErrorString(r));
    c->launches += 1;
  }
  std::vector<double> tot(o.W + 1);
  SGP_CUDA(c, cudaMemcpyAsync(tot.data(), o.dTotal, static_cast<size_t>(o.W + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  if (tot[o.W] != 0.0) return fail(c, err_code, err_msg);
  *val_out = tot[0];
  for (int i = 1; i < o.W; ++i) grad_out[i - 1] = tot[i];
  return SGP_OK;
}
}  // namespace

int sgp_bcm_nll(sgp_ctx* h, const sgp_kernel_desc* k, const sgp_hyper* hypers, int32_t nh, double* nll_out,
                double* grad_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!nll_out || (nh > 0 && !grad_out)) return fail(c, SGP_E_BADARG, "sgp_bcm_nll: null output");
  SGP_CUDA(c, cudaSetDevice(c->device));
  ObjectiveArgs o;
  int rc = objective_setup(c, k, hypers, nh, o);
  if (rc != SGP_OK) return rc;
  // fast path: on-chip Cholesky per expert (SPD kernel matrices of <= 168 points -- every default configuration).
  // general path: experts of any size, or a kernel matrix on which Cholesky broke down (not positive definite): the
  // reference's own arithmetic, LU with partial pivoting and log|det| with the sign dropped (logDetAndInv.scala:36-63,
  // GPR:59), on kernel matrices staged in global memory.  The choice is rank-local; the one all-reduce per evaluation
  // happens afterwards on every rank.
  bool general = bcm_nll_smem_bytes(c->ex_nmax) > 227 * 1024;
  if (!general) {
    SGP_CUDA(c, launch_bcm_nll(c->dEx, c->dEy, c->dEoff, c->n_experts, c->ex_d, c->ex_nmax, o.kf, o.dBeta, nh, o.dKind,
                               o.dTerm, o.dDim, o.dCoef, o.dValue, o.any_ard, c->dNllPer, o.dTotal, o.dFlags, c->stream));
    c->launches += 2;
    int flags = 0;
    SGP_CUDA(c, cudaMemcpyAsync(&flags, o.dFlags, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    SGP_CUDA(c, cudaStreamSynchronize(c->stream));
    general = (flags & 1) != 0;
  }
  c->bcm_general = general;
  if (general) {
    rc = ctx_scratch(c, c->bcm_ws, bcm_general_workspace_bytes(c->n_experts, c->ex_nmax));
    if (rc != SGP_OK) return rc;
    SGP_CUDA(c, cudaMemsetAsync(o.dFlags, 0, sizeof(int), c->stream));
    int blas_status = 0;
    SGP_CUDA(c, launch_bcm_nll_general(c->blas, &blas_status, c->bcm_ws.p, c->dEx, c->dEy, c->dEoff, c->n_experts, c->ex_d,
                                       c->ex_nmax, o.kf, o.dBeta, nh, o.dKind, o.dTerm, o.dDim, o.dCoef, o.dValue,
                                       o.any_ard, c->dNllPer, o.dTotal, o.dFlags, c->stream));
    if (blas_status != 0) return fail(c, SGP_E_CUDA, "cuBLAS batched LU failed, status " + std::to_string(blas_status));
    c->launches += 5;
  }
  return objective_finish(c, o, nll_out, grad_out, 2, SGP_E_SINGULAR,
                          "an expert's kernel matrix is singular (MatrixSingularException, logDetAndInv.scala:27-28)");
}

int sgp_laplace_nll(sgp_ctx* h, const sgp_kernel_desc* k, const sgp_hyper* hypers, int32_t nh, double tol,
                    double* neg_log_z_out, double* grad_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!neg_log_z_out || (nh > 0 && !grad_out) || !(tol > 0.0)) return fail(c, SGP_E_BADARG, "sgp_laplace_nll: bad argument");
  SGP_CUDA(c, cudaSetDevice(c->device));
  ObjectiveArgs o;
  int rc = objective_setup(c, k, hypers, nh, o);
  if (rc != SGP_OK) return rc;
  if (laplace_smem_bytes(c->ex_nmax) > 227 * 1024)
    return fail(c, SGP_E_BADARG, "datasetSizeForExpert too large for the on-chip Laplace kernel (max 117 points per expert)");
  SGP_CUDA(c, launch_laplace(c->dEx, c->dEy, c->dEf, c->dEoff, c->n_experts, c->ex_d, c->ex_nmax, o.kf, o.dBeta, nh,
                             o.dKind, o.dTerm, o.dDim, o.dCoef, o.dValue, o.any_ard, tol, c->dNllPer, o.dTotal, o.dFlags, c->stream));
  c->launches += 2;
  return objective_finish(c, o, neg_log_z_out, grad_out, 1, SGP_E_NOT_PD,
                          "an expert's B = I + sqrt(W) K sqrt(W) is not positive definite (increase sigma2)");
}

int sgp_experts_get_f(sgp_ctx* h, double* f_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->dEf || !f_out) return fail(c, SGP_E_STATE, "sgp_experts_upload should have been called first");
  SGP_CUDA(c, cudaSetDevice(c->device));
  SGP_CUDA(c, cudaMemcpyAsync(f_out, c->dEf, static_cast<size_t>(c->ex_n) * 8, cudaMemcpyDeviceToHost, c->stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  return SGP_OK;
}

int sgp_last_path(const sgp_ctx* h) {
  const Ctx* c = reinterpret_cast<const Ctx*>(h);
  return c ? c->last_path : -1;
}

int sgp_last_bcm_path(const sgp_ctx* h) {
  const Ctx* c = reinterpret_cast<const Ctx*>(h);
  return c ? (c->bcm_general ? 1 : 0) : -1;
}

int sgp_last_tail_path(const sgp_ctx* h) {
  const Ctx* c = reinterpret_cast<const Ctx*>(h);
  if (!c || !c->has_magic_run) return -1;
  return c->tail_fast ? 1 : 0;
}

int sgp_debug_i8_tile(sgp_ctx* h, float* T_out, uint32_t* w_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  SGP_CUDA(c, cudaSetDevice(c->device));
  if (!c->dbgT) {   // arm: the next I8 launches dump the first distance tile of CTA (0,0)
    SGP_CUDA(c, cudaMalloc(&c->dbgT, 128 * 64 * 4));
    SGP_CUDA(c, cudaMalloc(&c->dbgW, 128 * 64 * 4));
    SGP_CUDA(c, cudaMemset(c->dbgT, 0, 128 * 64 * 4));
    SGP_CUDA(c, cudaMemset(c->dbgW, 0, 128 * 64 * 4));
    SGP_CUDA(c, cudaMalloc(&c->dbgClk, (2560 + 148 * 32) * 8));
    SGP_CUDA(c, cudaMemset(c->dbgClk, 0, (2560 + 148 * 32) * 8));
  }
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  if (T_out) SGP_CUDA(c, cudaMemcpy(T_out, c->dbgT, 128 * 64 * 4, cudaMemcpyDeviceToHost));
  if (w_out) SGP_CUDA(c, cudaMemcpy(w_out, c->dbgW, 128 * 64 * 4, cudaMemcpyDeviceToHost));
  return SGP_OK;
}

int sgp_debug_i8_timeline(sgp_ctx* h, long long* out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c || !out) return SGP_E_BADARG;
  if (!c->dbgClk) return fail(c, SGP_E_STATE, "arm with sgp_debug_i8_tile first");
  SGP_CUDA(c, cudaSetDevice(c->device));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  SGP_CUDA(c, cudaMemcpy(out, c->dbgClk, (2560 + 148 * 32) * 8, cudaMemcpyDeviceToHost));
  return SGP_OK;
}

int sgp_event_record(sgp_ctx* h, int slot) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (slot < 0 || slot >= 8) return fail(c, SGP_E_BADARG, "event slot out of range");
  SGP_CUDA(c, cudaSetDevice(c->device));
  if (!c->user_events[slot]) SGP_CUDA(c, cudaEventCreate(&c->user_events[slot]));
  SGP_CUDA(c, cudaEventRecord(c->user_events[slot], c->stream));
  return SGP_OK;
}

int sgp_event_elapsed_ms(sgp_ctx* h, int a, int b, double* ms) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (a < 0 || a >= 8 || b < 0 || b >= 8 || !ms || !c->user_events[a] || !c->user_events[b])
    return fail(c, SGP_E_BADARG, "bad event slots");
  SGP_CUDA(c, cudaSetDevice(c->device));
  SGP_CUDA(c, cudaEventSynchronize(c->user_events[b]));
  float f = 0.f;
  SGP_CUDA(c, cudaEventElapsedTime(&f, c->user_events[a], c->user_events[b]));
  *ms = f;
  return SGP_OK;
}

// One sweep launch over n device-resident points (prep of the fp16 operand images + the sweep kernel).
static int sweep_device(Ctx* c, const void* dX, int x_is_f32, long long n, float* dK) {
  const int nch = i8_nchunks(c->d);
  const size_t xb = i8_points_scratch_bytes(n, nch);
  const size_t yb = static_cast<size_t>((n + 63) / 64) * 64 * sizeof(float);
  if (xb > c->i8_xt_bytes) {
    SGP_CUDA(c, cudaStreamSynchronize(c->stream));
    cudaFree(c->dI8Xt); c->dI8Xt = nullptr; c->i8_xt_bytes = 0;
    SGP_CUDA(c, cudaMalloc(&c->dI8Xt, xb));
    c->i8_xt_bytes = xb;
  }
  if (yb > c->i8_ys_bytes) {
    SGP_CUDA(c, cudaStreamSynchronize(c->stream));
    cudaFree(c->dI8Ys); c->dI8Ys = nullptr; c->i8_ys_bytes = 0;
    SGP_CUDA(c, cudaMalloc(&c->dI8Ys, yb));
    c->i8_ys_bytes = yb;
  }
  SGP_CUDA(c, launch_i8_prep_points(c->dI8Xt, c->dI8Ys, dX, x_is_f32, nullptr, n, c->d, c->dI8Scale, c->dI8Centre, c->dI8Flags,
                                    c->dI8NormSum, nullptr, c->stream));
  SGP_CUDA(c, launch_kmn_sweep(c->dI8Xt, c->dI8Zt, n, c->d, c->m, c->m_pad, c->num_sms, c->kf.scale[0], dK, c->stream));
  c->launches += 2;
  return SGP_OK;
}

int sgp_kmn_sweep_device(sgp_ctx* h, const void* dX, int32_t x_is_f32, int64_t n, float* dK_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->begun) return fail(c, SGP_E_STATE, "setTrainingVectors method should have been called first");
  if (n <= 0 || !dX || !dK_out) return fail(c, SGP_E_BADARG, "null argument");
  if (!c->i8_ok) return fail(c, SGP_E_BADARG, "sgp_kmn_sweep needs a kernel with exactly one non-Eye term and d <= 32");
  SGP_CUDA(c, cudaSetDevice(c->device));
  return sweep_device(c, dX, x_is_f32, n, dK_out);
}

int sgp_kmn_sweep(sgp_ctx* h, const void* X, int32_t x_is_f32, int64_t n, float* K_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->begun) return fail(c, SGP_E_STATE, "setTrainingVectors method should have been called first");
  if (n <= 0 || !X || !K_out) return fail(c, SGP_E_BADARG, "null argument");
  if (!c->i8_ok) return fail(c, SGP_E_BADARG, "sgp_kmn_sweep needs a kernel with exactly one non-Eye term and d <= 32");
  SGP_CUDA(c, cudaSetDevice(c->device));
  const size_t esz = x_is_f32 ? 4 : 8;
  const long long chunk = 65536;
  const long long cn0 = n < chunk ? n : chunk;
  int rc = ctx_scratch(c, c->sweep_ws, static_cast<size_t>(cn0) * c->d * esz + static_cast<size_t>(cn0) * c->m * sizeof(float));
  if (rc != SGP_OK) return rc;
  float* dK = static_cast<float*>(c->sweep_ws.p);
  void* dX = dK + static_cast<size_t>(cn0) * c->m;
  for (long long p0 = 0; p0 < n; p0 += chunk) {
    const long long cn = (n - p0 < chunk) ? (n - p0) : chunk;
    SGP_CUDA(c, cudaMemcpyAsync(dX, static_cast<const char*>(X) + static_cast<size_t>(p0) * c->d * esz,
                                static_cast<size_t>(cn) * c->d * esz, cudaMemcpyHostToDevice, c->stream));
    rc = sweep_device(c, dX, x_is_f32, cn, dK);
    if (rc != SGP_OK) return rc;
    SGP_CUDA(c, cudaMemcpyAsync(K_out + static_cast<size_t>(p0) * c->m, dK, static_cast<size_t>(cn) * c->m * sizeof(float),
                                cudaMemcpyDeviceToHost, c->stream));
    SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  int flags = 0;
  SGP_CUDA(c, cudaMemcpy(&flags, c->dI8Flags, sizeof(int), cudaMemcpyDeviceToHost));
  if (flags & 1)
    return fail(c, SGP_E_RANGE, "scaled coordinates exceed the fp16 operand range of the tensor-core distance contraction; "
                                "use sgp_cross_kernel");
  return SGP_OK;
}

int sgp_greedy_active_set(sgp_ctx* h, const sgp_kernel_desc* k, const double* X, const double* y, int64_t n, int32_t d,
                          int64_t n_experts, int64_t first_index, int32_t m_target, int64_t* indices_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!k || !X || !y || !indices_out || n <= 0 || d <= 0 || m_target <= 0 || k->n_terms <= 0 || !k->terms)
    return fail(c, SGP_E_BADARG, "sgp_greedy_active_set: null or empty argument");
  if (n_experts <= 0) return fail(c, SGP_E_BADARG, "numberOfExperts == 0 (N < datasetSizeForExpert / 2)");
  if (first_index < 0 || first_index >= n) return fail(c, SGP_E_BADARG, "first_index out of range");
  if (n > 2147483647LL) return fail(c, SGP_E_BADARG, "sgp_greedy_active_set: n too large for one device");
  SGP_CUDA(c, cudaSetDevice(c->device));
  KernelFlat kf;
  std::vector<double> beta(static_cast<size_t>(kMaxTerms) * d, 0.0);
  for (int t = 0; t < k->n_terms; ++t) {
    const sgp_kernel_term& term = k->terms[t];
    if (!(term.scale >= 0.0)) return fail(c, SGP_E_BADARG, "requirement failed: C should be positive");
    kf.self_kernel += term.scale;
    if (term.type == SGP_TERM_EYE) { kf.eye_sum += term.scale; continue; }
    if (kf.n_terms == kMaxTerms) return fail(c, SGP_E_BADARG, "too many non-Eye kernel terms (max 4)");
    double* bt = beta.data() + static_cast<size_t>(kf.n_terms) * d;
    if (term.type == SGP_TERM_ARD) {
      if (!term.beta) return fail(c, SGP_E_BADARG, "ARD term without beta");
      for (int j = 0; j < d; ++j) bt[j] = term.beta[j];
    } else if (term.type == SGP_TERM_RBF) {
      if (!(term.sigma > 0.0)) return fail(c, SGP_E_BADARG, "RBF sigma must be > 0");
      for (int j = 0; j < d; ++j) bt[j] = 1.0 / (std::sqrt(2.0) * term.sigma);
    } else {
      return fail(c, SGP_E_BADARG, "unknown kernel term type");
    }
    kf.scale[kf.n_terms++] = term.scale;
  }
  static_assert(sizeof(long long) == sizeof(int64_t), "index type");
  return run_greedy(c, kf, beta, X, y, n, d, n_experts, first_index, m_target, reinterpret_cast<long long*>(indices_out));
}

int sgp_cross_kernel(sgp_ctx* h, const double* X, int64_t n, double* K_out) {
  Ctx* c = reinterpret_cast<Ctx*>(h);
  if (!c) return SGP_E_BADARG;
  if (!c->begun) return fail(c, SGP_E_STATE, "setTrainingVectors method should have been called first");
  if (n <= 0 || !X || !K_out) return fail(c, SGP_E_BADARG, "null argument");
  if (n > 65535 * 8) return fail(c, SGP_E_BADARG, "sgp_cross_kernel: n too large for one call");
  SGP_CUDA(c, cudaSetDevice(c->device));
  int rc = ctx_scratch(c, c->cross_ws, (static_cast<size_t>(n) * c->d + static_cast<size_t>(n) * c->m) * 8);
  if (rc != SGP_OK) return rc;
  double* dX = static_cast<double*>(c->cross_ws.p);
  double* dK = dX + static_cast<size_t>(n) * c->d;
  SGP_CUDA(c, cudaMemcpyAsync(dX, X, static_cast<size_t>(n) * c->d * 8, cudaMemcpyHostToDevice, c->stream));
  if (c->kf.n_terms > 0) {
    SGP_CUDA(c, launch_cross_kernel(dK, dX, c->dZs, c->dBeta, c->kf, n, c->d, c->dpad, c->m, c->m_pad, c->stream));
    c->launches += 1;
  } else {
    SGP_CUDA(c, cudaMemsetAsync(dK, 0, static_cast<size_t>(n) * c->m * 8, c->stream));
  }
  SGP_CUDA(c, cudaMemcpyAsync(K_out, dK, static_cast<size_t>(n) * c->m * 8, cudaMemcpyDeviceToHost, c->stream));
  SGP_CUDA(c, cudaStreamSynchronize(c->stream));
  return SGP_OK;
}

}  // extern "C"
