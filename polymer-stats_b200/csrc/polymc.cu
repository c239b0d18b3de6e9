// polymc.cu — host side of libpolymc_b200.so: the C ABI declared in include/polymc.h.
//
// No CPU fallback: every compute entry point needs a CUDA device and reports
// PMC_ERR_NO_DEVICE / PMC_ERR_CUDA otherwise.
#include "handle.h"
#include "exchange.cuh"

namespace {

thread_local std::string g_err;

// the FFI mirrors of pmc_case (ctypes in polymc/lib.py, the Julia struct in julia/polymc_host.jl) rely on it
static_assert(sizeof(pmc_case) == 13 * 8 + 2 * 8 + 6 * 4 + 4 * 8 + 4 * 4, "pmc_case layout changed: bump PMC_ABI_VERSION");

int fail(int code, const std::string& msg) { return pmc_fail(code, msg); }

}  // namespace

int pmc_fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

// ---- cache of device blocks ------------------------------------------------------------------------------------
namespace {
struct PoolBlock {
  void* ptr;
  size_t bytes;
  int device;
};
constexpr size_t kPoolCapBytes = (size_t)24 << 30;   // of the 180 GB per GPU
std::mutex g_pool_mu;
std::vector<PoolBlock> g_pool_free;                  // blocks waiting for reuse
std::unordered_map<void*, PoolBlock> g_pool_live;    // blocks handed out
}  // namespace

cudaError_t pmc_pool_alloc(void** ptr, size_t bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (bytes == 0) bytes = 1;
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    size_t best = g_pool_free.size();
    for (size_t k = 0; k < g_pool_free.size(); ++k) {   // best fit within 2× (a sweep asks for the same sizes again)
      const PoolBlock& b = g_pool_free[k];
      if (b.device == dev && b.bytes >= bytes && b.bytes <= 2 * bytes + 4096 &&
          (best == g_pool_free.size() || b.bytes < g_pool_free[best].bytes))
        best = k;
    }
    if (best != g_pool_free.size()) {
      const PoolBlock b = g_pool_free[best];
      g_pool_free.erase(g_pool_free.begin() + (long)best);
      g_pool_live[b.ptr] = b;
      *ptr = b.ptr;
      return cudaSuccess;
    }
  }
  e = cudaMalloc(ptr, bytes);
  if (e == cudaErrorMemoryAllocation) {  // give the cache back and try once more
    cudaGetLastError();
    pmc_release_cached_memory();
    e = cudaMalloc(ptr, bytes);
  }
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lk(g_pool_mu);
  g_pool_live[*ptr] = PoolBlock{*ptr, bytes, dev};
  return cudaSuccess;
}

void pmc_pool_free(void* ptr) {
  if (!ptr) return;
  std::lock_guard<std::mutex> lk(g_pool_mu);
  auto it = g_pool_live.find(ptr);
  if (it == g_pool_live.end()) {  // not ours
    cudaFree(ptr);
    return;
  }
  const PoolBlock b = it->second;
  g_pool_live.erase(it);
  size_t held = 0;
  for (const PoolBlock& f : g_pool_free) held += f.bytes;
  if (held + b.bytes > kPoolCapBytes) {  // the cache is bounded: beyond the cap a block goes straight back to the driver
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(b.device);
    cudaFree(b.ptr);
    cudaSetDevice(cur);
    return;
  }
  g_pool_free.push_back(b);
}

extern "C" int32_t pmc_release_cached_memory(void) {
  std::vector<PoolBlock> blocks;
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    blocks.swap(g_pool_free);
  }
  int cur = 0;
  cudaGetDevice(&cur);
  for (const PoolBlock& b : blocks) {
    cudaSetDevice(b.device);
    cudaFree(b.ptr);
  }
  cudaSetDevice(cur);
  return PMC_OK;
}

namespace {

int ensure_scratch(pmc_handle* h, size_t doubles) {
  if (h->scratch_cap >= doubles) return PMC_OK;
  if (h->scratch) pmc_pool_free(h->scratch);
  h->scratch = nullptr;
  h->scratch_cap = 0;
  PMC_CU(pool_alloc(&h->scratch, doubles * sizeof(double)));
  h->scratch_cap = doubles;
  return PMC_OK;
}

int check_handle(const pmc_handle* h) {
  if (!h) return fail(PMC_ERR_INVALID, "null handle");
  cudaError_t e = cudaSetDevice(h->device);
  if (e != cudaSuccess) return fail(PMC_ERR_NO_DEVICE, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  return PMC_OK;
}

int check_chain(const pmc_handle* h, int64_t chain) {
  if (chain < 0 || chain >= h->nchains) return fail(PMC_ERR_INVALID, "chain index out of range");
  return PMC_OK;
}

// Launch pick(std::integral_constant<int, T>) at the planned block size T of the CTA helper kernels.
template <class Pick, class Args>
static int launch_cta_kernel(pmc_handle* h, Pick pick, int nblocks, size_t smem, const Args& a) {
  return with<32, 64, 128, 256, 512>(plan_run(h).cta_threads,
                                     [&](auto T) { return launch(h, pick(T), nblocks, T, smem, a); });
}

int launch_energy(pmc_handle* h, const EnergyArgs& a, int nblocks) {
  return launch_cta_kernel(h, [](auto t) { return k_energy_cta<decltype(t)::value>; }, nblocks, cta_smem_bytes(h->n), a);
}

// ΔU of one scripted move with the rectangle precision the run kernel of this handle uses.
int launch_delta_cta(pmc_handle* h, const DeltaArgs& a) {
  const RunPlan p = plan_run(h);
  if (!p.f32) return launch_cta_kernel(h, [](auto t) { return k_delta_cta<decltype(t)::value>; }, 1, cta_smem_bytes(h->n), a);
  return with<64, 128, 256, 512>(p.cta_threads, [&](auto T) {
    return launch(h, k_delta_cta<T, 1>, 1, T, ((cta_smem_bytes(h->n) + 15) & ~(size_t)15) + f32_smem_bytes(h->n), a);
  });
}

int launch_reinit(pmc_handle* h, const ReinitArgs& a) {
  return launch_cta_kernel(h, [](auto t) { return k_reinit_cta<decltype(t)::value>; }, (int)h->nchains,
                           cta_smem_bytes(h->n), a);
}

// Recompute the running scalars of every chain from its records (re-synchronisation).
int refresh(pmc_handle* h, bool rebind_gauge, int first = 0, int count = -1) {
  h->dyn_fresh = h->dynx_fresh = false;
  EnergyArgs a{};
  a.mono = h->mono; a.par = h->par; a.dyn = h->dyn;
  a.out4 = nullptr; a.obs6 = nullptr;
  a.n = h->n; a.energy_type = h->energy_type; a.first_chain = first;
  a.update_dyn = 1; a.rebind_gauge = rebind_gauge ? 1 : 0;
  a.dynx = h->dynx; a.out8 = nullptr;
  return launch_energy(h, a, count < 0 ? (int)h->nchains : count);
}

int validate_case(const pmc_case& c, const pmc_case& first) {
  if (c.n < 1) return fail(PMC_ERR_INVALID, "num-monomers must be >= 1");
  if (c.n != first.n || c.energy_type != first.energy_type)
    return fail(PMC_ERR_INVALID, "all cases of one handle must share num-monomers and energy-type; bucket the sweep");
  if (c.chain_type != PMC_CHAIN_DIELECTRIC && c.chain_type != PMC_CHAIN_POLAR)
    return fail(PMC_ERR_INVALID, "chain-type is not understood.");  // eap_chain.jl:86
  if (c.energy_type < 0 || c.energy_type > 3)
    return fail(PMC_ERR_INVALID, "energy-type is not understood.");  // eap_chain.jl:104
  if (!(c.kT > 0.0)) return fail(PMC_ERR_INVALID, "kT must be positive");
  if (c.accum_mode != 0 && c.accum_mode != 1) return fail(PMC_ERR_INVALID, "accum_mode must be 0 or 1");
  if (c.clustering && c.n < 2) return fail(PMC_ERR_INVALID, "the clustering driver needs num-monomers >= 2");
  if (c.planar != first.planar) return fail(PMC_ERR_INVALID, "all cases of one handle must be planar or none");
  if (c.planar && (!c.clustering || c.kappa != 0.0 || c.energy_type == PMC_ENERGY_CUTOFF || c.do_flips))
    return fail(PMC_ERR_INVALID, "the 2-D tree has only the clustering driver, without bending, cut-off or --do-flips");
  if (!(c.cluster_prob >= 0.0 && c.cluster_prob <= 1.0) && c.clustering)
    return fail(PMC_ERR_INVALID, "cluster-prob must be in [0,1]");
  return PMC_OK;
}

// Does this case need the composite-trial kernels (cluster flips, bending energy, cut-off pair sum)?
bool needs_cluster_path(const pmc_case& c) {
  return c.clustering != 0 || c.kappa != 0.0 || c.energy_type == PMC_ENERGY_CUTOFF;
}

ChainParams params_of(const pmc_case& c0, double kT_scale = 1.0) {
  pmc_case c = c0;
  c.kT = c0.kT * kT_scale;  // burn-in stage temperature (mcmc_clustering_eap_chain.jl:367-381)
  ChainParams P{};
  if (c.chain_type == PMC_CHAIN_DIELECTRIC) {  // dipole_response.jl:7-11
    P.alpha = (c.K1 - c.K2) * c.E0;
    P.beta = c.K2 * c.E0;
    P.m = 0.0;
    P.gauge0 = -(c.K1 + 2 * c.K2) * c.E0 * c.E0 * (double)c.n / (3 * c.kT);  // average.jl:109-112
  } else {  // dipole_response.jl:27-29 with M = mu·I (eap_chain.jl:84)
    P.alpha = 0.0;
    P.beta = 0.0;
    P.m = c.mu;
    P.gauge0 = -c.mu * c.E0 * (double)c.n / (3 * c.kT);  // average.jl:114-118, eigvals(mu·I)[end] = mu
  }
  P.E0 = c.E0; P.kT = c.kT; P.inv_kT = 1.0 / c.kT;
  P.Fz = c.Fz; P.Fx = c.Fx; P.b = c.b;
  P.adj_lb = c.adj_lb; P.adj_ub = c.adj_ub; P.adj_scale = c.adj_scale;
  P.cF = 0.2 + 0.8 * std::exp(-(c.Fx * c.Fx + c.Fz * c.Fz) / c.kT);
  P.phi_step0 = c.phi_step; P.theta_step0 = c.theta_step;
  P.steps_per_adjust = c.steps_per_adjust;
  P.do_flips = c.do_flips; P.umbrella = c.umbrella; P.force_init = c.force_init;
  P.kappa = c.kappa; P.psi0 = c.psi0;
  P.crad2 = (c.cutoff_radius * c.b) * (c.cutoff_radius * c.b);  // UCutoff(cutoff-radius·mlen), eap_chain.jl:102
  P.cluster_prob = c.cluster_prob;
  P.clustering = c.clustering; P.alpha_carry = c.alpha_carry; P.cutoff_full = c.cutoff_full;
  P.planar = c.planar;
  return P;
}

int fetch_dyn(pmc_handle* h) {
  if (h->dyn_fresh && h->host_dyn.size() == (size_t)h->nchains) return PMC_OK;  // averages + accumulators + diagnostics: one copy
  h->host_dyn.resize((size_t)h->nchains);
  PMC_CU(cudaMemcpyAsync(h->host_dyn.data(), h->dyn, sizeof(ChainDyn) * (size_t)h->nchains, cudaMemcpyDeviceToHost,
                         h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  h->dyn_fresh = true;
  return PMC_OK;
}

}  // namespace

extern "C" {

int32_t pmc_abi_version(void) { return PMC_ABI_VERSION; }

const char* pmc_last_error(void) { return g_err.c_str(); }

int32_t pmc_device_count(int32_t* count) {
  if (!count) return fail(PMC_ERR_INVALID, "null count");
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess) {
    cudaGetLastError();
    *count = 0;
    return fail(PMC_ERR_NO_DEVICE, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
  }
  *count = c;
  return PMC_OK;
}

int32_t pmc_create(const pmc_case* cases, int64_t ncases, int32_t replicas_per_case, uint64_t seed, int32_t device,
                   uint32_t chain_id_base, pmc_handle** out) {
  if (!out) return fail(PMC_ERR_INVALID, "null out handle");
  *out = nullptr;
  if (!cases || ncases < 1 || replicas_per_case < 1) return fail(PMC_ERR_INVALID, "need >= 1 case and >= 1 replica");
  for (int64_t i = 0; i < ncases; ++i) {
    int rc = validate_case(cases[i], cases[0]);
    if (rc) return rc;
  }
  const int64_t nchains = ncases * (int64_t)replicas_per_case;
  if (nchains > (int64_t)0x7fffffff) return fail(PMC_ERR_INVALID, "too many chains for one handle");
  const bool trace = env_int("PMC_TRACE_CREATE", 0) != 0;   // developer timing of the set-up phases, to stderr
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!trace) return;
    const auto t = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[pmc_create] %-22s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t - t_prev).count());
    t_prev = t;
  };
  int ndev = 0;
  {
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1) {
      cudaGetLastError();
      return fail(PMC_ERR_NO_DEVICE, "no CUDA device available (libpolymc_b200 has no CPU fallback)");
    }
  }
  if (device < 0 || device >= ndev) return fail(PMC_ERR_NO_DEVICE, "device index out of range");
  PMC_CU(cudaSetDevice(device));
  const int n = (int)cases[0].n;
  if (cases[0].n > 1 << 20) return fail(PMC_ERR_UNSUPPORTED, "num-monomers too large");
  if (cta_smem_bytes(n) > (size_t)kSmemMax)
    return fail(PMC_ERR_UNSUPPORTED, "chain too long: x and mu of one chain must fit one CTA's 227 KB shared memory "
                                     "(num-monomers <= ~4100)");
  pmc_handle* h = new (std::nothrow) pmc_handle();
  if (!h) return fail(PMC_ERR_NOMEM, "host allocation failed");
  h->device = device;
  h->nchains = nchains;
  h->n = n;
  h->energy_type = cases[0].energy_type;
  h->seed = seed;
  h->chain_id_base = chain_id_base;
  {
    int sms = 0;  // (cudaGetDeviceProperties costs tens of milliseconds; one attribute is all that is needed)
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) h->sm_count = sms;
  }
  h->compensated = 0;
  for (int64_t i = 0; i < ncases; ++i)
    if (cases[i].accum_mode || cases[i].umbrella) h->compensated = 1;  // umbrella weights span many decades
  h->cases.assign(cases, cases + ncases);
  h->replicas = replicas_per_case;
  h->planar = cases[0].planar;
  for (int64_t i = 0; i < ncases; ++i)
    if (needs_cluster_path(cases[i])) h->cluster_mode = 1;
  const bool cta_pairs = h->energy_type == PMC_ENERGY_INTERACTING || h->energy_type == PMC_ENERGY_CUTOFF;
  if (h->cluster_mode && cta_pairs && cluster_delta_smem_bytes(n, plan_run(h).cta_threads) > (size_t)kSmemMax) {
    delete h;
    return fail(PMC_ERR_UNSUPPORTED, "chain too long for the clustering / bending / cut-off kernels: 18 n doubles "
                                     "must fit one CTA's 227 KB shared memory (num-monomers <= ~1570)");
  }

  lap("validate + handle");
  std::vector<ChainParams> par((size_t)nchains);
  std::vector<ChainDyn> dyn((size_t)nchains);
  for (int64_t c = 0; c < nchains; ++c) {
    const pmc_case& cs = cases[c / replicas_per_case];
    par[(size_t)c] = params_of(cs);
    ChainDyn d{};
    d.phi_step = cs.phi_step;
    d.theta_step = cs.theta_step;
    dyn[(size_t)c] = d;
  }
  auto cleanup = [&](int rc) {
    pmc_destroy(h);
    return rc;
  };
#define PMC_TRY(expr)                    \
  do {                                   \
    int rc__ = [&]() -> int {            \
      expr;                              \
      return PMC_OK;                     \
    }();                                 \
    if (rc__) return cleanup(rc__);      \
  } while (0)
  lap("host tables");
  const size_t total = (size_t)nchains * (size_t)n;
  PMC_TRY(PMC_CU(pool_alloc(&h->mono, total * sizeof(MonoRec))));
  PMC_TRY(PMC_CU(pool_alloc(&h->par, (size_t)nchains * sizeof(ChainParams))));
  PMC_TRY(PMC_CU(pool_alloc(&h->dyn, (size_t)nchains * sizeof(ChainDyn))));
  PMC_TRY(PMC_CU(pool_alloc(&h->dynx, (size_t)nchains * sizeof(ChainDynX))));
  PMC_TRY(PMC_CU(cudaMemset(h->dynx, 0, (size_t)nchains * sizeof(ChainDynX))));
  PMC_TRY(PMC_CU(pool_alloc(&h->flags, (size_t)nchains * sizeof(int))));
  PMC_TRY(PMC_CU(cudaEventCreate(&h->ev0)));
  PMC_TRY(PMC_CU(cudaEventCreate(&h->ev1)));
  lap("cudaMalloc + events");
  PMC_TRY(PMC_CU(cudaMemcpy(h->par, par.data(), (size_t)nchains * sizeof(ChainParams), cudaMemcpyHostToDevice)));
  PMC_TRY(PMC_CU(cudaMemcpy(h->dyn, dyn.data(), (size_t)nchains * sizeof(ChainDyn), cudaMemcpyHostToDevice)));
  lap("H2D par + dyn");
  {
    const int tb = 256;
    const long long blocks = ((long long)total + tb - 1) / tb;
    k_fill_random<<<(unsigned)blocks, tb, 0, h->stream>>>(h->mono, (long long)total, n, seed, chain_id_base, 0u,
                                                          h->planar);
    ++h->launches;
    PMC_TRY(PMC_CU(cudaGetLastError()));
  }
  {
    int rc = refresh(h, /*rebind_gauge=*/true);
    if (rc) return cleanup(rc);
  }
  PMC_TRY(PMC_CU(cudaStreamSynchronize(h->stream)));
  lap("fill + energies");
#undef PMC_TRY
  *out = h;
  return PMC_OK;
}

void pmc_destroy(pmc_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);  // nothing in flight may still use blocks that return to the cache
  if (h->mono) pmc_pool_free(h->mono);
  if (h->cand) pmc_pool_free(h->cand);
  if (h->par) pmc_pool_free(h->par);
  if (h->dyn) pmc_pool_free(h->dyn);
  if (h->dynx) pmc_pool_free(h->dynx);
  if (h->state) pmc_pool_free(h->state);
  if (h->x0buf) pmc_pool_free(h->x0buf);
  if (h->traj) pmc_pool_free(h->traj);
  if (h->roll) pmc_pool_free(h->roll);
  if (h->scratch) pmc_pool_free(h->scratch);
  if (h->flags) pmc_pool_free(h->flags);
  if (h->pair_work) pmc_pool_free(h->pair_work);
  if (h->pair_order) pmc_pool_free(h->pair_order);
  if (h->pair_next) pmc_pool_free(h->pair_next);
  for (void* p : {(void*)h->ex_pairs, (void*)h->ex_stats, (void*)h->ex_walker, (void*)h->ex_wstate, (void*)h->ex_trips,
                  (void*)h->tt_out[0], (void*)h->tt_out[1], (void*)h->tt_out[2]})
    if (p) pmc_pool_free(p);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  delete h;
}

int64_t pmc_num_chains(const pmc_handle* h) { return h ? h->nchains : 0; }
int64_t pmc_num_monomers(const pmc_handle* h) { return h ? h->n : 0; }

int32_t pmc_set_ensemble_hint(pmc_handle* h, int64_t ensemble_chains) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (ensemble_chains < 0) return fail(PMC_ERR_INVALID, "ensemble_chains must be >= 0");
  h->shape_chains = ensemble_chains;
  return PMC_OK;
}

int32_t pmc_set_pair_precision(pmc_handle* h, int32_t mode) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (mode != PMC_PAIR_FP64 && mode != PMC_PAIR_FP32) return fail(PMC_ERR_INVALID, "pair precision must be PMC_PAIR_FP64 or PMC_PAIR_FP32");
  h->pair_precision = mode;
  return PMC_OK;
}

int32_t pmc_pair_precision(const pmc_handle* h) { return h && plan_run(h).f32 ? PMC_PAIR_FP32 : PMC_PAIR_FP64; }

int32_t pmc_block_threads(const pmc_handle* h) { return h ? plan_run(h).cta_threads : 0; }

int32_t pmc_set_stream(pmc_handle* h, void* cuda_stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  PMC_CU(cudaStreamSynchronize(h->stream));
  h->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  return PMC_OK;
}

static int set_state_range(pmc_handle* h, int64_t first, int64_t count, const double* phi, const double* theta) {
  if (!phi || !theta) return fail(PMC_ERR_INVALID, "null state pointer");
  const size_t m = (size_t)count * (size_t)h->n;
  int rc = ensure_scratch(h, 2 * m);
  if (rc) return rc;
  PMC_CU(cudaMemcpyAsync(h->scratch, phi, m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  PMC_CU(cudaMemcpyAsync(h->scratch + m, theta, m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  const int tb = 256;
  k_build_records<<<(unsigned)((m + tb - 1) / tb), tb, 0, h->stream>>>(h->mono + (size_t)first * h->n, h->scratch,
                                                                         h->scratch + m, (long long)m, h->planar);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  // a new state replaces the chain the weight function was built from (mcmc_eap_chain.jl:175-177)
  rc = refresh(h, /*rebind_gauge=*/true, (int)first, (int)count);
  if (rc) return rc;
  PMC_CU(cudaStreamSynchronize(h->stream));
  return PMC_OK;
}

static int get_state_range(pmc_handle* h, int64_t first, int64_t count, double* phi, double* theta) {
  if (!phi || !theta) return fail(PMC_ERR_INVALID, "null state pointer");
  const size_t m = (size_t)count * (size_t)h->n;
  int rc = ensure_scratch(h, 2 * m);
  if (rc) return rc;
  const int tb = 256;
  k_extract_state<<<(unsigned)((m + tb - 1) / tb), tb, 0, h->stream>>>(h->mono + (size_t)first * h->n, h->scratch,
                                                                         h->scratch + m, (long long)m);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  PMC_CU(cudaMemcpyAsync(phi, h->scratch, m * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaMemcpyAsync(theta, h->scratch + m, m * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  return PMC_OK;
}

int32_t pmc_set_state(pmc_handle* h, int64_t chain, const double* phi, const double* theta) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_chain(h, chain))) return rc;
  return set_state_range(h, chain, 1, phi, theta);
}

int32_t pmc_get_state(pmc_handle* h, int64_t chain, double* phi, double* theta) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_chain(h, chain))) return rc;
  return get_state_range(h, chain, 1, phi, theta);
}

int32_t pmc_set_state_all(pmc_handle* h, const double* phi, const double* theta) {
  int rc = check_handle(h);
  if (rc) return rc;
  return set_state_range(h, 0, h->nchains, phi, theta);
}

int32_t pmc_get_state_all(pmc_handle* h, double* phi, double* theta) {
  int rc = check_handle(h);
  if (rc) return rc;
  return get_state_range(h, 0, h->nchains, phi, theta);
}

static int energy_range(pmc_handle* h, int64_t first, int64_t count, double* out4, double* obs6,
                        double* out8 = nullptr) {
  int rc = ensure_scratch(h, (size_t)count * 18);
  if (rc) return rc;
  EnergyArgs a{};
  a.mono = h->mono; a.par = h->par; a.dyn = h->dyn;
  a.out4 = h->scratch;
  a.obs6 = h->scratch + (size_t)count * 4;
  a.out8 = h->scratch + (size_t)count * 10;
  a.dynx = nullptr;
  a.n = h->n; a.energy_type = h->energy_type; a.first_chain = (int)first;
  a.update_dyn = 0; a.rebind_gauge = 0;
  rc = launch_energy(h, a, (int)count);
  if (rc) return rc;
  if (out4)
    PMC_CU(cudaMemcpyAsync(out4, a.out4, (size_t)count * 4 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (obs6)
    PMC_CU(cudaMemcpyAsync(obs6, a.obs6, (size_t)count * 6 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (out8)
    PMC_CU(cudaMemcpyAsync(out8, a.out8, (size_t)count * 8 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  return PMC_OK;
}

static int launch_delta_segment(pmc_handle* h, const SegDeltaArgs& a) {
  const bool cta_pairs = h->energy_type == PMC_ENERGY_INTERACTING || h->energy_type == PMC_ENERGY_CUTOFF;
  if (cta_pairs) return launch_delta_segment_cta(h, a);
  if (h->energy_type == PMC_ENERGY_ISING) k_delta_segment_lane<true><<<1, 32, 0, h->stream>>>(a);
  else k_delta_segment_lane<false><<<1, 32, 0, h->stream>>>(a);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  return PMC_OK;
}

static int fetch_dynx(pmc_handle* h) {
  if (h->dynx_fresh && h->host_dynx.size() == (size_t)h->nchains) return PMC_OK;
  h->host_dynx.resize((size_t)h->nchains);
  PMC_CU(cudaMemcpyAsync(h->host_dynx.data(), h->dynx, sizeof(ChainDynX) * (size_t)h->nchains, cudaMemcpyDeviceToHost,
                         h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  h->dynx_fresh = true;
  return PMC_OK;
}

int32_t pmc_energy(pmc_handle* h, int64_t chain, double out[4]) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_chain(h, chain))) return rc;
  if (!out) return fail(PMC_ERR_INVALID, "null out");
  return energy_range(h, chain, 1, out, nullptr);
}

int32_t pmc_energy_all(pmc_handle* h, double* out) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!out) return fail(PMC_ERR_INVALID, "null out");
  return energy_range(h, 0, h->nchains, out, nullptr);
}

int32_t pmc_observables(pmc_handle* h, int64_t chain, double out[6]) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_chain(h, chain))) return rc;
  if (!out) return fail(PMC_ERR_INVALID, "null out");
  return energy_range(h, chain, 1, nullptr, out);
}

int32_t pmc_delta_u(pmc_handle* h, int64_t chain, int64_t idx0, double dphi, double dtheta, double out[3]) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_chain(h, chain))) return rc;
  if (!out) return fail(PMC_ERR_INVALID, "null out");
  if (idx0 < 0 || idx0 >= h->n) return fail(PMC_ERR_INVALID, "monomer index out of range");
  if (h->cluster_mode) {  // bending energy / cut-off pair sum live in the composite-trial code
    double o[12];
    rc = pmc_delta_segment(h, chain, idx0, dphi, dtheta, 0, idx0, idx0, o);
    if (rc) return rc;
    MonoRec rec;
    PMC_CU(cudaMemcpy(&rec, h->mono + (size_t)chain * h->n + idx0, sizeof(rec), cudaMemcpyDeviceToHost));
    const double traw = rec.theta + dtheta;
    out[0] = o[0]; out[1] = o[1]; out[2] = (traw < 0.0 || traw > kPi) ? 1.0 : 0.0;
    return PMC_OK;
  }
  if ((rc = ensure_scratch(h, 8))) return rc;
  DeltaArgs a{};
  a.mono = h->mono; a.par = h->par; a.out = h->scratch;
  a.n = h->n; a.energy_type = h->energy_type; a.chain = (int)chain; a.idx = (int)idx0;
  a.dphi = dphi; a.dtheta = dtheta;
  if (h->energy_type == PMC_ENERGY_INTERACTING) {
    if ((rc = launch_delta_cta(h, a))) return rc;
  } else {
    k_delta_lane<<<1, 32, 0, h->stream>>>(a);
    ++h->launches;
    PMC_CU(cudaGetLastError());
  }
  double tmp[4];
  PMC_CU(cudaMemcpyAsync(tmp, h->scratch, sizeof(tmp), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  out[0] = tmp[0]; out[1] = tmp[1]; out[2] = tmp[2];
  return PMC_OK;
}

int64_t pmc_rows_for(const pmc_handle* h, int64_t nsteps, int64_t stepout) {
  if (!h || stepout <= 0 || nsteps <= 0) return 0;
  // all chains share the step counter (same number of pmc_run trials since the last init)
  const int64_t step0 = h->host_dyn.empty() ? 0 : (int64_t)h->host_dyn[0].step;
  return (step0 + nsteps) / stepout - step0 / stepout;
}

// The MCMC kernel of this handle as planned now (plan_run), followed, for the FP32 rectangle, by the energy refresh: the
// running energy is the sum of FP32-rounded ΔU of the accepted moves; put it back on the exact energy of the chain after
// every launch (one FP64 energy evaluation per chain ≈ three trials' worth of pairs).
static int dispatch_run(pmc_handle* h, const RunArgs& a) {
  const RunPlan p = plan_run(h);
  int rc;
  switch (p.family) {
    case RunFamily::cta_win:
    case RunFamily::cta_win_spec: rc = launch_run_cta(h, p, a); break;
    case RunFamily::cta_pair: rc = launch_run_pair(h, p, a); break;
    case RunFamily::lane:
    case RunFamily::warp: rc = launch_run_lane(h, p, a); break;
    case RunFamily::cta_cluster:
    case RunFamily::cta_cluster_spec: rc = launch_run_cluster_cta(h, p, a); break;
    default: rc = launch_run_cluster_lane(h, p, a); break;
  }
  if (rc) return rc;
  return p.f32 ? refresh(h, /*rebind_gauge=*/false) : PMC_OK;
}

static int run_impl(pmc_handle* h, int64_t nsteps, int64_t stepout, double* traj, double* roll, int roll_cols,
                    double* state);

int32_t pmc_run(pmc_handle* h, int64_t nsteps, int64_t stepout, double* traj, double* roll) {
  return run_impl(h, nsteps, stepout, traj, roll, 17, nullptr);
}

int32_t pmc_run_ex(pmc_handle* h, int64_t nsteps, int64_t stepout, double* traj, double* roll19, double* state) {
  if (h && !h->cluster_mode)
    return fail(PMC_ERR_INVALID, "pmc_run_ex needs a clustering-driver handle (clustering, bend-mod or cutoff case)");
  return run_impl(h, nsteps, stepout, traj, roll19, 19, state);
}

// The shared step counter (one copy, so the row counts of the next launches are known on the host).
static int fetch_step0(pmc_handle* h) {
  ChainDyn d0;
  PMC_CU(cudaMemcpyAsync(&d0, h->dyn, sizeof(ChainDyn), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  if (h->host_dyn.empty()) h->host_dyn.resize((size_t)h->nchains);
  h->host_dyn[0] = d0;
  return PMC_OK;
}

static int grow(double** buf, size_t* cap, size_t doubles) {
  if (doubles <= *cap) return PMC_OK;
  if (*buf) pmc_pool_free(*buf);
  *buf = nullptr; *cap = 0;
  PMC_CU(pool_alloc(buf, doubles * sizeof(double)));
  *cap = doubles;
  return PMC_OK;
}

// Device row buffers of one launch of `rows` rows and the launch arguments of the run kernels.
static int run_args(pmc_handle* h, int64_t nsteps, int64_t stepout, int64_t rows, int roll_cols, bool want_state,
                    RunArgs& a) {
  const size_t ntraj = (size_t)h->nchains * (size_t)rows * 8, nroll = (size_t)h->nchains * (size_t)rows * roll_cols;
  const size_t nstate = want_state ? (size_t)h->nchains * (size_t)rows * 2 * (size_t)h->n : 0;
  int rc;
  if ((rc = grow(&h->state, &h->state_cap, nstate))) return rc;
  if ((rc = grow(&h->traj, &h->traj_cap, ntraj))) return rc;
  if ((rc = grow(&h->roll, &h->roll_cap, nroll))) return rc;
  a = RunArgs{};
  a.mono = h->mono; a.par = h->par; a.dyn = h->dyn;
  a.traj = h->traj; a.roll = h->roll;
  a.nsteps = nsteps; a.stepout = stepout; a.rows = rows;
  a.seed = h->seed; a.chain_id_base = h->chain_id_base;
  a.n = h->n; a.nchains = (int)h->nchains; a.energy_type = h->energy_type;
  a.dynx = h->dynx; a.state = nstate ? h->state : nullptr; a.roll_cols = roll_cols;
  a.compensated = h->compensated;
  // k_run_warp_cluster: trials per window.  An accepted trial invalidates the later trials of the window that read its
  // segment and every invalidation costs a serial re-evaluation pass, but the per-window work (draws, prefix sums,
  // averagers) is amortised over the window: 32 wins from n = 25 to 400 (profiles/r01f_tune_warp_cluster.txt).
  a.window = 32;
  return PMC_OK;
}

static int run_impl(pmc_handle* h, int64_t nsteps, int64_t stepout, double* traj, double* roll, int roll_cols,
                    double* state) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (nsteps < 0) return fail(PMC_ERR_INVALID, "nsteps must be >= 0");
  if (nsteps == 0) return PMC_OK;
  if (nsteps >= (1LL << 40)) return fail(PMC_ERR_INVALID, "nsteps must stay below 2^40");
  // re-synchronise running scalars against a full recompute (records drift, SURVEY §7 "hard parts")
  if ((rc = refresh(h, false))) return rc;
  // step0 (shared by all chains) decides the row count
  if ((rc = fetch_step0(h))) return rc;
  const int64_t rows = pmc_rows_for(h, nsteps, stepout);
  const size_t ntraj = (size_t)h->nchains * (size_t)rows * 8, nroll = (size_t)h->nchains * (size_t)rows * roll_cols;
  const size_t nstate = state ? (size_t)h->nchains * (size_t)rows * 2 * (size_t)h->n : 0;
  RunArgs a;
  if ((rc = run_args(h, nsteps, stepout, rows, roll_cols, state != nullptr, a))) return rc;
  PMC_CU(cudaEventRecord(h->ev0, h->stream));
  if ((rc = dispatch_run(h, a))) return rc;
  PMC_CU(cudaEventRecord(h->ev1, h->stream));
  if (traj && rows > 0)
    PMC_CU(cudaMemcpyAsync(traj, h->traj, ntraj * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (roll && rows > 0)
    PMC_CU(cudaMemcpyAsync(roll, h->roll, nroll * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (state && rows > 0)
    PMC_CU(cudaMemcpyAsync(state, h->state, nstate * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  PMC_CU(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
  h->host_dyn[0].step += nsteps;
  return PMC_OK;
}

int32_t pmc_last_run_ms(const pmc_handle* h, float* ms) {
  if (!h || !ms) return fail(PMC_ERR_INVALID, "null argument");
  *ms = h->last_ms;
  return PMC_OK;
}

int64_t pmc_launch_count(const pmc_handle* h) { return h ? h->launches : 0; }

int32_t pmc_kernel_name(pmc_handle* h, char* buf, int32_t buflen) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!buf || buflen < 1) return fail(PMC_ERR_INVALID, "null or empty name buffer");
  const RunPlan p = plan_run(h);
  if (p.smem > (size_t)kSmemMax) return fail(PMC_ERR_UNSUPPORTED, "chain too long for this kernel's shared memory");
  std::snprintf(buf, (size_t)buflen, "%s", kernel_name(p).c_str());
  return PMC_OK;
}

int32_t pmc_reinit(pmc_handle* h, int32_t* replaced) {
  int rc = check_handle(h);
  if (rc) return rc;
  const size_t total = (size_t)h->nchains * (size_t)h->n;
  if (!h->cand) PMC_CU(pool_alloc(&h->cand, total * sizeof(MonoRec)));
  h->init += 1;
  const int tb = 256;
  k_fill_random<<<(unsigned)((total + tb - 1) / tb), tb, 0, h->stream>>>(h->cand, (long long)total, h->n, h->seed,
                                                                        h->chain_id_base, (uint32_t)h->init, h->planar);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  if ((rc = refresh(h, false))) return rc;  // current U, Ω exact before comparing
  ReinitArgs a{};
  a.mono = h->mono; a.cand = h->cand; a.par = h->par; a.dyn = h->dyn; a.replaced = h->flags;
  a.seed = h->seed; a.chain_id_base = h->chain_id_base;
  a.n = h->n; a.energy_type = h->energy_type; a.new_init = h->init;
  if ((rc = launch_reinit(h, a))) return rc;
  if (h->cluster_mode && (rc = refresh(h, false))) return rc;  // Σψ, Σcos²θ of the new chains
  if (replaced)
    PMC_CU(cudaMemcpyAsync(replaced, h->flags, (size_t)h->nchains * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  if (!h->host_dyn.empty()) h->host_dyn[0].step = 0;
  return PMC_OK;
}

int32_t pmc_averages(pmc_handle* h, double* avg, double* acc_rate, double* normalizer) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = fetch_dyn(h))) return rc;
  for (int64_t c = 0; c < h->nchains; ++c) {
    const ChainDyn& d = h->host_dyn[(size_t)c];
    const double nrm = d.acc[16] + d.comp[16];
    if (avg)
      for (int k = 0; k < 16; ++k) avg[c * 16 + k] = (d.acc[k] + d.comp[k]) / nrm;  // get_avg, average.jl:38
    if (acc_rate) acc_rate[c] = d.steps_total ? (double)d.nacc_total / (double)d.steps_total : 0.0;
    if (normalizer) normalizer[c] = nrm;
  }
  return PMC_OK;
}

int32_t pmc_accumulators(pmc_handle* h, double* sums) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!sums) return fail(PMC_ERR_INVALID, "null sums");
  if ((rc = fetch_dyn(h))) return rc;
  for (int64_t c = 0; c < h->nchains; ++c) {
    const ChainDyn& d = h->host_dyn[(size_t)c];
    for (int k = 0; k < kNumAcc; ++k) sums[c * kNumAcc + k] = d.acc[k] + d.comp[k];
  }
  return PMC_OK;
}

int32_t pmc_diagnostics(pmc_handle* h, double* diag) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!diag) return fail(PMC_ERR_INVALID, "null diag");
  if ((rc = fetch_dyn(h))) return rc;
  for (int64_t c = 0; c < h->nchains; ++c) {
    const ChainDyn& d = h->host_dyn[(size_t)c];
    double* o = diag + c * 8;
    o[0] = d.phi_step; o[1] = d.theta_step;
    o[2] = (double)d.nacc; o[3] = (double)d.natt;
    o[4] = (double)d.nacc_total; o[5] = (double)d.steps_total;
    o[6] = d.U; o[7] = d.drift_max;
  }
  return PMC_OK;
}

int32_t pmc_energy_ex(pmc_handle* h, int64_t chain, double out[8]) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_chain(h, chain))) return rc;
  if (!out) return fail(PMC_ERR_INVALID, "null out");
  return energy_range(h, chain, 1, nullptr, nullptr, out);
}

int32_t pmc_delta_segment(pmc_handle* h, int64_t chain, int64_t idx0, double dphi, double dtheta, int32_t reflect,
                          int64_t lo0, int64_t hi0, double out[12]) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_chain(h, chain))) return rc;
  if (!out) return fail(PMC_ERR_INVALID, "null out");
  if (idx0 < 0 || idx0 >= h->n) return fail(PMC_ERR_INVALID, "monomer index out of range");
  if (reflect && !(0 <= lo0 && lo0 <= idx0 && idx0 <= hi0 && hi0 < h->n))
    return fail(PMC_ERR_INVALID, "cluster bounds must satisfy 0 <= lo <= idx <= hi < n");
  if ((rc = ensure_scratch(h, 16))) return rc;
  SegDeltaArgs a{};
  a.mono = h->mono; a.par = h->par; a.out = h->scratch;
  a.n = h->n; a.energy_type = h->energy_type; a.chain = (int)chain; a.idx = (int)idx0;
  a.lo = (int)lo0; a.hi = (int)hi0; a.reflect = reflect ? 1 : 0;
  a.dphi = dphi; a.dtheta = dtheta;
  if ((rc = launch_delta_segment(h, a))) return rc;
  PMC_CU(cudaMemcpyAsync(out, h->scratch, 12 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  return PMC_OK;
}

int32_t pmc_begin_stage(pmc_handle* h, double kT_scale) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!(kT_scale > 0.0)) return fail(PMC_ERR_INVALID, "kT_scale must be positive");
  h->kT_scale = kT_scale;
  std::vector<ChainParams> par((size_t)h->nchains);
  for (int64_t c = 0; c < h->nchains; ++c) par[(size_t)c] = params_of(h->cases[(size_t)(c / h->replicas)], kT_scale);
  PMC_CU(cudaMemcpyAsync(h->par, par.data(), par.size() * sizeof(ChainParams), cudaMemcpyHostToDevice, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));  // `par` is pageable host memory
  h->init += 1;
  if (h->planar) {  // 2D/mcmc_clustering_eap_chain.jl:151: `chain = EAPChain(pargs)` — every stage builds a new chain
    const size_t total = (size_t)h->nchains * (size_t)h->n;
    k_fill_random<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(h->mono, (long long)total, h->n, h->seed,
                                                                          h->chain_id_base, (uint32_t)h->init, 1);
    ++h->launches;
    PMC_CU(cudaGetLastError());
  }
  const int tb = 128;
  k_begin_stage<<<(unsigned)((h->nchains + tb - 1) / tb), tb, 0, h->stream>>>(h->dyn, h->dynx, h->par, (int)h->nchains,
                                                                             h->init);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  if ((rc = refresh(h, /*rebind_gauge=*/true))) return rc;  // chain.U = U(chain); wf = AntiDipoleWeightFunction(chain)
  PMC_CU(cudaStreamSynchronize(h->stream));
  if (!h->host_dyn.empty()) h->host_dyn[0].step = 0;
  return PMC_OK;
}

int32_t pmc_init_x0(pmc_handle* h, const double* x0, int64_t x0_len, const double dx0[2]) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!x0 || !dx0) return fail(PMC_ERR_INVALID, "null x0/dx0");
  if (h->planar) return fail(PMC_ERR_UNSUPPORTED, "the 2-D tree has no --x0 (2D/inc/eap_chain.jl:66-67)");
  if (x0_len != 2 && x0_len != 2 * (int64_t)h->n) return fail(PMC_ERR_INVALID, "Invalid input for 'x0'");  // eap_chain.jl:76
  if (!h->x0buf) PMC_CU(pool_alloc(&h->x0buf, 2 * (size_t)h->n * sizeof(double)));
  PMC_CU(cudaMemcpyAsync(h->x0buf, x0, (size_t)x0_len * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  const size_t total = (size_t)h->nchains * (size_t)h->n;
  const int tb = 256;
  k_fill_x0<<<(unsigned)((total + tb - 1) / tb), tb, 0, h->stream>>>(h->mono, (long long)total, h->n, h->seed,
                                                                    h->chain_id_base, 0u, h->x0buf, (int)x0_len, dx0[0],
                                                                    dx0[1]);
  ++h->launches;
  PMC_CU(cudaGetLastError());
  if ((rc = refresh(h, /*rebind_gauge=*/true))) return rc;
  PMC_CU(cudaStreamSynchronize(h->stream));
  return PMC_OK;
}

int32_t pmc_extra_accumulators(pmc_handle* h, double* sums) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!sums) return fail(PMC_ERR_INVALID, "null sums");
  if ((rc = fetch_dynx(h))) return rc;
  for (int64_t c = 0; c < h->nchains; ++c) {
    const ChainDynX& d = h->host_dynx[(size_t)c];
    sums[c * 2 + 0] = d.acc[0] + d.comp[0];
    sums[c * 2 + 1] = d.acc[1] + d.comp[1];
  }
  return PMC_OK;
}

int32_t pmc_extra_averages(pmc_handle* h, double* ex) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!ex) return fail(PMC_ERR_INVALID, "null ex");
  if ((rc = fetch_dyn(h))) return rc;
  if ((rc = fetch_dynx(h))) return rc;
  for (int64_t c = 0; c < h->nchains; ++c) {
    const ChainDynX& d = h->host_dynx[(size_t)c];
    const ChainDyn& D = h->host_dyn[(size_t)c];
    const double nrm = D.acc[16] + D.comp[16];
    ex[c * 2 + 0] = (d.acc[0] + d.comp[0]) / nrm;
    ex[c * 2 + 1] = (d.acc[1] + d.comp[1]) / nrm;
  }
  return PMC_OK;
}

int32_t pmc_cluster_stats(pmc_handle* h, double* out) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!out) return fail(PMC_ERR_INVALID, "null out");
  if ((rc = fetch_dynx(h))) return rc;
  for (int64_t c = 0; c < h->nchains; ++c) {
    const ChainDynX& d = h->host_dynx[(size_t)c];
    out[c * 3 + 0] = d.ncluster; out[c * 3 + 1] = d.cluster_sum; out[c * 3 + 2] = d.cluster_max;
  }
  return PMC_OK;
}

// ---- replica exchange ---------------------------------------------------------------------------------------
namespace {

// PMC_CU that yields the status instead of returning it (for clean-up on failure)
int cu_rc(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return PMC_OK;
  cudaGetLastError();
  return fail(e == cudaErrorMemoryAllocation ? PMC_ERR_NOMEM : PMC_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define PMC_CU_RC(expr) cu_rc((expr), #expr)

void ladder_clear(pmc_handle* h) {
  for (void* p : {(void*)h->ex_pairs, (void*)h->ex_stats, (void*)h->ex_walker, (void*)h->ex_wstate, (void*)h->ex_trips})
    if (p) pmc_pool_free(p);
  h->ex_pairs = nullptr; h->ex_stats = nullptr; h->ex_walker = nullptr; h->ex_wstate = nullptr; h->ex_trips = nullptr;
  h->ex_count[0] = h->ex_count[1] = 0;
  h->ex_round = 0;
  h->ladder.clear();
}

// The name of the first field in which two rungs of one ladder differ although it enters the energy or the target
// density, or nullptr.
const char* rung_mismatch(const pmc_case& x, const pmc_case& y) {
#define PMC_SAME(f) if (x.f != y.f) return #f;
  PMC_SAME(E0) PMC_SAME(K1) PMC_SAME(K2) PMC_SAME(mu) PMC_SAME(b) PMC_SAME(n) PMC_SAME(chain_type) PMC_SAME(energy_type)
  PMC_SAME(kappa) PMC_SAME(psi0) PMC_SAME(cutoff_radius) PMC_SAME(cutoff_full) PMC_SAME(clustering) PMC_SAME(planar)
#undef PMC_SAME
  return nullptr;
}

// One round: the pairs of parity round & 1 of every ladder and replica column.
int exchange_round(pmc_handle* h) {
  const int parity = (int)(h->ex_round & 1);
  ExchangeArgs a{};
  a.mono = h->mono; a.par = h->par; a.dyn = h->dyn; a.dynx = h->dynx;
  a.pairs = h->ex_pairs + (parity ? h->ex_count[0] : 0);
  a.stats = h->ex_stats; a.walker = h->ex_walker; a.wstate = h->ex_wstate; a.trips = h->ex_trips;
  a.accepted = h->flags;
  a.seed = h->seed; a.chain_id_base = h->chain_id_base; a.n = h->n; a.round = h->ex_round;
  int rc = launch_exchange(h, a, h->ex_count[parity]);
  if (rc) return rc;
  h->ex_round += 1;
  h->dyn_fresh = h->dynx_fresh = false;
  return PMC_OK;
}

int tempering_impl(pmc_handle* h, int64_t nsteps, int64_t every, int64_t stepout, double* traj, double* roll,
                   int roll_cols, double* state) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (h->ladder.empty()) return fail(PMC_ERR_INVALID, "no ladders set (pmc_set_ladders)");
  if (nsteps < 0) return fail(PMC_ERR_INVALID, "nsteps must be >= 0");
  if (nsteps == 0) return PMC_OK;
  if (nsteps >= (1LL << 40)) return fail(PMC_ERR_INVALID, "nsteps must stay below 2^40");
  if (every < 1 || nsteps % every != 0) return fail(PMC_ERR_INVALID, "exchange_every must divide nsteps");
  if (stepout > 0 && every % stepout != 0) return fail(PMC_ERR_INVALID, "stepout must divide exchange_every, or be 0");
  if ((rc = fetch_step0(h))) return rc;   // the only copy to the host before the results
  const int64_t rows_total = pmc_rows_for(h, nsteps, stepout), rows = stepout > 0 ? every / stepout : 0;
  const size_t per_row[3] = {8, (size_t)roll_cols, 2 * (size_t)h->n};
  double* host_out[3] = {traj, roll, state};
  for (int k = 0; k < 3; ++k)
    if (host_out[k] && rows_total > 0 &&
        (rc = grow(&h->tt_out[k], &h->tt_cap[k], (size_t)h->nchains * (size_t)rows_total * per_row[k])))
      return rc;
  RunArgs a;
  if ((rc = run_args(h, every, stepout, rows, roll_cols, state != nullptr, a))) return rc;
  const double* chunk_out[3] = {h->traj, h->roll, h->state};
  PMC_CU(cudaEventRecord(h->ev0, h->stream));
  for (int64_t k = 0; k < nsteps / every; ++k) {   // exactly pmc_run(every) followed by pmc_exchange, k times
    if ((rc = refresh(h, false))) return rc;
    if ((rc = dispatch_run(h, a))) return rc;
    for (int j = 0; j < 3; ++j)
      if (host_out[j] && rows > 0 &&
          (rc = launch_place_rows(h, h->tt_out[j], chunk_out[j], rows, rows_total, k * rows, (int)per_row[j])))
        return rc;
    if ((rc = exchange_round(h))) return rc;
  }
  PMC_CU(cudaEventRecord(h->ev1, h->stream));
  for (int k = 0; k < 3; ++k)
    if (host_out[k] && rows_total > 0)
      PMC_CU(cudaMemcpyAsync(host_out[k], h->tt_out[k], (size_t)h->nchains * (size_t)rows_total * per_row[k] * sizeof(double),
                             cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  PMC_CU(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
  h->host_dyn[0].step += nsteps;
  return PMC_OK;
}

}  // namespace

int32_t pmc_set_ladders(pmc_handle* h, const int32_t* rungs, int64_t len) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (len < 0 || (len > 0 && !rungs)) return fail(PMC_ERR_INVALID, "null or negative-length rung list");
  const int64_t ncases = (int64_t)h->cases.size(), R = h->replicas;
  std::vector<std::vector<int32_t>> ladders(1);
  for (int64_t i = 0; i < len; ++i) {
    if (rungs[i] == -1) {
      if (ladders.back().empty()) return fail(PMC_ERR_INVALID, "empty ladder in the rung list");
      if (i + 1 < len) ladders.emplace_back();
      continue;
    }
    if (rungs[i] < 0 || rungs[i] >= ncases) return fail(PMC_ERR_INVALID, "rung " + std::to_string(rungs[i]) +
                                                                             " is not a case index of this handle");
    ladders.back().push_back(rungs[i]);
  }
  if (len == 0) ladders.clear();
  std::vector<char> seen((size_t)ncases, 0);
  for (const auto& L : ladders) {
    if (L.size() < 2) return fail(PMC_ERR_INVALID, "a ladder needs at least two rungs");
    for (int32_t c : L) {
      if (seen[(size_t)c]) return fail(PMC_ERR_INVALID, "case " + std::to_string(c) + " appears more than once in the ladders");
      seen[(size_t)c] = 1;
      const pmc_case& x = h->cases[(size_t)c];
      const pmc_case& y = h->cases[(size_t)L[0]];
      if (x.umbrella) return fail(PMC_ERR_INVALID, "umbrella sampling cannot be tempered: its weights depend on kT and F");
      if (const char* f = rung_mismatch(x, y))
        return fail(PMC_ERR_INVALID, std::string("rungs of one ladder must agree on ") + f + " (cases " +
                                         std::to_string(L[0]) + " and " + std::to_string(c) + ")");
      if (x.energy_type == PMC_ENERGY_CUTOFF && !x.cutoff_full && (x.Fz != y.Fz || x.Fx != y.Fx))
        return fail(PMC_ERR_INVALID, "a force ladder needs F in the energy: the cut-off energy without cutoff_full has no -r.F");
    }
  }
  // pairs of even rounds first, then those of odd rounds; both lists are walked in ladder, rung, replica order
  std::vector<ExPair> pairs[2];
  std::vector<int> wstate((size_t)h->nchains, 0);
  for (const auto& L : ladders) {
    const int m = (int)L.size();
    for (int64_t r = 0; r < R; ++r) wstate[(size_t)(L[0] * R + r)] = 1;
    for (int i = 0; i + 1 < m; ++i)
      for (int64_t r = 0; r < R; ++r)
        pairs[i & 1].push_back(ExPair{(int)(L[i] * R + r), (int)(L[i + 1] * R + r), L[i],
                                      (i == 0 ? 1 : 0) | (i + 2 == m ? 2 : 0)});
  }
  ladder_clear(h);
  if (ladders.empty()) return PMC_OK;
  const size_t c = (size_t)h->nchains, np = pairs[0].size() + pairs[1].size();
  std::vector<long long> walker(c);
  for (size_t i = 0; i < c; ++i) walker[i] = (long long)h->chain_id_base + (long long)i;
  pairs[0].insert(pairs[0].end(), pairs[1].begin(), pairs[1].end());
  auto undo = [&](int code) { ladder_clear(h); return code; };
  if ((rc = PMC_CU_RC(pool_alloc(&h->ex_pairs, np * sizeof(ExPair))))) return undo(rc);
  if ((rc = PMC_CU_RC(pool_alloc(&h->ex_stats, (size_t)ncases * 2 * sizeof(unsigned long long))))) return undo(rc);
  if ((rc = PMC_CU_RC(pool_alloc(&h->ex_walker, c * sizeof(long long))))) return undo(rc);
  if ((rc = PMC_CU_RC(pool_alloc(&h->ex_wstate, c * sizeof(int))))) return undo(rc);
  if ((rc = PMC_CU_RC(pool_alloc(&h->ex_trips, c * sizeof(long long))))) return undo(rc);
  if ((rc = PMC_CU_RC(cudaMemcpyAsync(h->ex_pairs, pairs[0].data(), np * sizeof(ExPair), cudaMemcpyHostToDevice, h->stream))) ||
      (rc = PMC_CU_RC(cudaMemsetAsync(h->ex_stats, 0, (size_t)ncases * 2 * sizeof(unsigned long long), h->stream))) ||
      (rc = PMC_CU_RC(cudaMemcpyAsync(h->ex_walker, walker.data(), c * sizeof(long long), cudaMemcpyHostToDevice, h->stream))) ||
      (rc = PMC_CU_RC(cudaMemcpyAsync(h->ex_wstate, wstate.data(), c * sizeof(int), cudaMemcpyHostToDevice, h->stream))) ||
      (rc = PMC_CU_RC(cudaMemsetAsync(h->ex_trips, 0, c * sizeof(long long), h->stream))) ||
      (rc = PMC_CU_RC(cudaStreamSynchronize(h->stream))))   // the host vectors are pageable and local
    return undo(rc);
  h->ex_count[0] = (int64_t)(np - pairs[1].size());
  h->ex_count[1] = (int64_t)pairs[1].size();
  h->ladder.assign(rungs, rungs + len);
  return PMC_OK;
}

int32_t pmc_exchange(pmc_handle* h, int32_t* accepted) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (h->ladder.empty()) return fail(PMC_ERR_INVALID, "no ladders set (pmc_set_ladders)");
  PMC_CU(cudaMemsetAsync(h->flags, 0, (size_t)h->nchains * sizeof(int), h->stream));
  if ((rc = exchange_round(h))) return rc;
  if (accepted)
    PMC_CU(cudaMemcpyAsync(accepted, h->flags, (size_t)h->nchains * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  return PMC_OK;
}

int32_t pmc_run_tempering(pmc_handle* h, int64_t nsteps, int64_t exchange_every, int64_t stepout, double* traj,
                          double* roll) {
  return tempering_impl(h, nsteps, exchange_every, stepout, traj, roll, 17, nullptr);
}

int32_t pmc_run_tempering_ex(pmc_handle* h, int64_t nsteps, int64_t exchange_every, int64_t stepout, double* traj,
                             double* roll19, double* state) {
  if (h && !h->cluster_mode)
    return fail(PMC_ERR_INVALID, "pmc_run_tempering_ex needs a clustering-driver handle (clustering, bend-mod or cutoff case)");
  return tempering_impl(h, nsteps, exchange_every, stepout, traj, roll19, 19, state);
}

int32_t pmc_exchange_stats(pmc_handle* h, double* pair_stats, int64_t* walker, int64_t* round_trips) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (h->ladder.empty()) return fail(PMC_ERR_INVALID, "no ladders set (pmc_set_ladders)");
  const size_t ncases = h->cases.size(), c = (size_t)h->nchains;
  std::vector<unsigned long long> st(ncases * 2);
  PMC_CU(cudaMemcpyAsync(st.data(), h->ex_stats, st.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
  static_assert(sizeof(long long) == sizeof(int64_t), "walker labels are 64-bit");
  if (walker) PMC_CU(cudaMemcpyAsync(walker, h->ex_walker, c * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  if (round_trips) PMC_CU(cudaMemcpyAsync(round_trips, h->ex_trips, c * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaStreamSynchronize(h->stream));
  if (pair_stats)
    for (size_t i = 0; i < st.size(); ++i) pair_stats[i] = (double)st[i];
  return PMC_OK;
}

// ---- checkpoint / resume ---------------------------------------------------------------------------------
namespace {
struct CkptHeader {
  uint64_t magic;        // "PMCCKPT3"
  int32_t abi, n, energy_type, cluster_mode, planar, init;
  int64_t nchains;
  uint64_t seed;
  uint32_t chain_id_base, pad;
  double kT_scale;
  int64_t host_step;
};
constexpr uint64_t kCkptMagic = 0x3354504b43434d50ull;
// Trailing block of a handle with ladders: this header, the rung list (int32), the pair statistics ([ncases][2] uint64),
// the walker labels (int64), the round-trip states (int32) and counts (int64) of every chain.
struct LadderHeader {
  uint64_t magic;        // "PMCLADR1"
  int64_t len, ncases, nchains, round;
};
constexpr uint64_t kLadderMagic = 0x315244414c434d50ull;

size_t ckpt_base_bytes(const pmc_handle* h) {
  const size_t c = (size_t)h->nchains;
  return sizeof(CkptHeader) + c * (size_t)h->n * sizeof(MonoRec) + c * sizeof(ChainDyn) + c * sizeof(ChainDynX);
}

size_t ladder_block_bytes(const pmc_handle* h) {
  if (h->ladder.empty()) return 0;
  const size_t c = (size_t)h->nchains;
  return sizeof(LadderHeader) + h->ladder.size() * sizeof(int32_t) + h->cases.size() * 2 * sizeof(unsigned long long) +
         c * (sizeof(long long) + sizeof(int) + sizeof(long long));
}
}  // namespace

int64_t pmc_checkpoint_bytes(const pmc_handle* h) {
  if (!h) return 0;
  return (int64_t)(ckpt_base_bytes(h) + ladder_block_bytes(h));
}

int32_t pmc_checkpoint_save(pmc_handle* h, void* buf, int64_t bytes) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!buf || bytes < pmc_checkpoint_bytes(h)) return fail(PMC_ERR_INVALID, "checkpoint buffer too small");
  CkptHeader hd{};
  hd.magic = kCkptMagic; hd.abi = PMC_ABI_VERSION; hd.n = h->n; hd.energy_type = h->energy_type;
  hd.cluster_mode = h->cluster_mode; hd.planar = h->planar; hd.init = h->init; hd.nchains = h->nchains;
  hd.seed = h->seed; hd.chain_id_base = h->chain_id_base; hd.kT_scale = h->kT_scale;
  hd.host_step = h->host_dyn.empty() ? 0 : (int64_t)h->host_dyn[0].step;
  unsigned char* p = static_cast<unsigned char*>(buf);
  std::memcpy(p, &hd, sizeof(hd));
  p += sizeof(hd);
  const size_t c = (size_t)h->nchains, nm = c * (size_t)h->n * sizeof(MonoRec);
  PMC_CU(cudaMemcpyAsync(p, h->mono, nm, cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaMemcpyAsync(p + nm, h->dyn, c * sizeof(ChainDyn), cudaMemcpyDeviceToHost, h->stream));
  PMC_CU(cudaMemcpyAsync(p + nm + c * sizeof(ChainDyn), h->dynx, c * sizeof(ChainDynX), cudaMemcpyDeviceToHost, h->stream));
  if (!h->ladder.empty()) {
    unsigned char* q = static_cast<unsigned char*>(buf) + ckpt_base_bytes(h);
    const LadderHeader lh{kLadderMagic, (int64_t)h->ladder.size(), (int64_t)h->cases.size(), h->nchains, h->ex_round};
    std::memcpy(q, &lh, sizeof(lh));
    q += sizeof(lh);
    std::memcpy(q, h->ladder.data(), h->ladder.size() * sizeof(int32_t));
    q += h->ladder.size() * sizeof(int32_t);
    const size_t ns = h->cases.size() * 2 * sizeof(unsigned long long);
    PMC_CU(cudaMemcpyAsync(q, h->ex_stats, ns, cudaMemcpyDeviceToHost, h->stream));
    q += ns;
    PMC_CU(cudaMemcpyAsync(q, h->ex_walker, c * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    q += c * sizeof(long long);
    PMC_CU(cudaMemcpyAsync(q, h->ex_wstate, c * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    q += c * sizeof(int);
    PMC_CU(cudaMemcpyAsync(q, h->ex_trips, c * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
  }
  PMC_CU(cudaStreamSynchronize(h->stream));
  return PMC_OK;
}

int32_t pmc_checkpoint_load(pmc_handle* h, const void* buf, int64_t bytes) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!buf || bytes < (int64_t)sizeof(CkptHeader)) return fail(PMC_ERR_INVALID, "checkpoint buffer too small");
  CkptHeader hd;
  std::memcpy(&hd, buf, sizeof(hd));
  if (hd.magic != kCkptMagic || hd.abi != PMC_ABI_VERSION) return fail(PMC_ERR_INVALID, "not a checkpoint of this ABI version");
  if (hd.n != h->n || hd.nchains != h->nchains || hd.energy_type != h->energy_type || hd.cluster_mode != h->cluster_mode ||
      hd.planar != h->planar || hd.seed != h->seed || hd.chain_id_base != h->chain_id_base)
    return fail(PMC_ERR_INVALID, "checkpoint belongs to a different ensemble (n, chains, energy type, seed or chain ids differ)");
  if (bytes < (int64_t)ckpt_base_bytes(h)) return fail(PMC_ERR_INVALID, "truncated checkpoint");
  const unsigned char* p = static_cast<const unsigned char*>(buf) + sizeof(hd);
  const size_t c = (size_t)h->nchains, nm = c * (size_t)h->n * sizeof(MonoRec);
  // the ladder block, validated before anything is loaded
  const unsigned char* q = static_cast<const unsigned char*>(buf) + ckpt_base_bytes(h);
  LadderHeader lh{};
  if (bytes >= (int64_t)(ckpt_base_bytes(h) + sizeof(lh))) std::memcpy(&lh, q, sizeof(lh));
  if (h->ladder.empty() && lh.magic == kLadderMagic)
    return fail(PMC_ERR_INVALID, "checkpoint holds replica-exchange ladders; set the same ladders before loading it");
  if (!h->ladder.empty()) {
    if (lh.magic != kLadderMagic) return fail(PMC_ERR_INVALID, "checkpoint has no replica-exchange ladders; this handle has");
    if (bytes < pmc_checkpoint_bytes(h)) return fail(PMC_ERR_INVALID, "truncated checkpoint");
    if (lh.len != (int64_t)h->ladder.size() || lh.ncases != (int64_t)h->cases.size() || lh.nchains != h->nchains ||
        std::memcmp(q + sizeof(lh), h->ladder.data(), h->ladder.size() * sizeof(int32_t)) != 0)
      return fail(PMC_ERR_INVALID, "checkpoint ladders differ from this handle's (pmc_set_ladders)");
  }
  if (hd.kT_scale != h->kT_scale) {  // the stage temperature lives in the per-chain constants
    std::vector<ChainParams> par(c);
    for (size_t i = 0; i < c; ++i) par[i] = params_of(h->cases[i / (size_t)h->replicas], hd.kT_scale);
    PMC_CU(cudaMemcpyAsync(h->par, par.data(), c * sizeof(ChainParams), cudaMemcpyHostToDevice, h->stream));
    PMC_CU(cudaStreamSynchronize(h->stream));
    h->kT_scale = hd.kT_scale;
  }
  PMC_CU(cudaMemcpyAsync(h->mono, p, nm, cudaMemcpyHostToDevice, h->stream));
  PMC_CU(cudaMemcpyAsync(h->dyn, p + nm, c * sizeof(ChainDyn), cudaMemcpyHostToDevice, h->stream));
  PMC_CU(cudaMemcpyAsync(h->dynx, p + nm + c * sizeof(ChainDyn), c * sizeof(ChainDynX), cudaMemcpyHostToDevice, h->stream));
  if (!h->ladder.empty()) {
    q += sizeof(lh) + h->ladder.size() * sizeof(int32_t);
    const size_t ns = h->cases.size() * 2 * sizeof(unsigned long long);
    PMC_CU(cudaMemcpyAsync(h->ex_stats, q, ns, cudaMemcpyHostToDevice, h->stream));
    q += ns;
    PMC_CU(cudaMemcpyAsync(h->ex_walker, q, c * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    q += c * sizeof(long long);
    PMC_CU(cudaMemcpyAsync(h->ex_wstate, q, c * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    q += c * sizeof(int);
    PMC_CU(cudaMemcpyAsync(h->ex_trips, q, c * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    h->ex_round = lh.round;
  }
  PMC_CU(cudaStreamSynchronize(h->stream));
  h->init = hd.init;
  h->dyn_fresh = h->dynx_fresh = false;
  if (h->host_dyn.empty()) h->host_dyn.resize(c);
  h->host_dyn[0].step = hd.host_step;
  return PMC_OK;
}

int32_t pmc_accumulators_dd(pmc_handle* h, double* hi, double* lo) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!hi || !lo) return fail(PMC_ERR_INVALID, "null hi/lo");
  if ((rc = fetch_dyn(h))) return rc;
  if ((rc = fetch_dynx(h))) return rc;
  auto two_sum = [](double a, double b, double& s, double& e) {  // renormalise: s + e = a + b exactly, |e| <= ulp(s)/2
    s = a + b;
    const double bb = s - a;
    e = (a - (s - bb)) + (b - bb);
  };
  for (int64_t c = 0; c < h->nchains; ++c) {
    const ChainDyn& d = h->host_dyn[(size_t)c];
    const ChainDynX& x = h->host_dynx[(size_t)c];
    for (int k = 0; k < kNumAcc; ++k) two_sum(d.acc[k], d.comp[k], hi[c * 19 + k], lo[c * 19 + k]);
    for (int k = 0; k < 2; ++k) two_sum(x.acc[k], x.comp[k], hi[c * 19 + 17 + k], lo[c * 19 + 17 + k]);
  }
  return PMC_OK;
}

int32_t pmc_fp64_peak_probe(int32_t device, int32_t iters, double* tflops, float* ms) {
  if (!tflops) return fail(PMC_ERR_INVALID, "null tflops");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    cudaGetLastError();
    return fail(PMC_ERR_NO_DEVICE, "no CUDA device available");
  }
  if (device < 0 || device >= ndev) return fail(PMC_ERR_NO_DEVICE, "device index out of range");
  PMC_CU(cudaSetDevice(device));
  if (iters < 1) iters = 1 << 16;
  cudaDeviceProp prop;
  PMC_CU(cudaGetDeviceProperties(&prop, device));
  double* sink = nullptr;
  PMC_CU(cudaMalloc(&sink, sizeof(double)));
  cudaEvent_t e0, e1;
  PMC_CU(cudaEventCreate(&e0));
  PMC_CU(cudaEventCreate(&e1));
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  k_fp64_probe<<<blocks, threads>>>(sink, 1024, 1.0000001, 1e-9);  // warm-up
  PMC_CU(cudaEventRecord(e0));
  k_fp64_probe<<<blocks, threads>>>(sink, iters, 1.0000001, 1e-9);
  PMC_CU(cudaEventRecord(e1));
  PMC_CU(cudaEventSynchronize(e1));
  PMC_CU(cudaGetLastError());
  float t = 0.f;
  PMC_CU(cudaEventElapsedTime(&t, e0, e1));
  const double flops = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
  *tflops = flops / ((double)t * 1e-3) / 1e12;
  if (ms) *ms = t;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  return PMC_OK;
}

}  // extern "C"
