// capi.cc — extern "C" boundary (include/towr_b200.h).  Owns device memory for
// the structure-class tables and the per-batch staging buffers.  There is no
// CPU evaluation path: without a CUDA device twb_batch_create fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/towr_b200.h"
#include "formulation.h"
#include "launch.h"

namespace {
// TWB_PROFILE=1: serialise every kernel on one stream, time each with events, print a table at exit
struct ProfRec { std::string label; cudaEvent_t a, b; };
std::vector<ProfRec> g_prof;
cudaEvent_t g_prof_last = nullptr;
bool g_prof_on = false;
void ProfHook(const char* label, cudaStream_t stream) {
  cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, stream);
  if (std::string(label) != "begin" && g_prof_last) g_prof.push_back({label, g_prof_last, e});
  g_prof_last = e;
}
void ProfReport() {
  cudaDeviceSynchronize();
  std::vector<std::pair<std::string, std::pair<double, int>>> agg;
  for (auto& r : g_prof) {
    float ms = 0; if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) continue;
    bool found = false;
    for (auto& a : agg) if (a.first == r.label) { a.second.first += ms; a.second.second++; found = true; }
    if (!found) agg.push_back({r.label, {ms, 1}});
  }
  for (auto& a : agg) std::fprintf(stderr, "[twb profile] %-14s n=%5d  avg %8.2f us\n", a.first.c_str(), a.second.second, 1e3 * a.second.first / a.second.second);
}
thread_local std::string g_err;
int Fail(int code, const std::string& why) { g_err = why; return code; }
int CudaFail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return TWB_ERR_CUDA;
}
template <class T>
cudaError_t Upload(const std::vector<T>& h, const T** d, std::vector<void*>* owned) {
  *d = nullptr;
  if (h.empty()) return cudaSuccess;
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, h.size() * sizeof(T));
  if (e != cudaSuccess) return e;
  owned->push_back(p);
  e = cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
  *d = static_cast<const T*>(p);
  return e;
}
}  // namespace

struct twb_problem {
  twb::Formulation f;
};

struct twb_batch {
  const twb_problem* prob = nullptr;
  int B = 0, device = 0;
  size_t ld = 0;                  // instances padded to a multiple of 32 (whole tiles of XT)
  twb::Plan plan{};
  std::vector<void*> owned;       // device allocations of the tables
  int* d_terrain = nullptr;       // per-instance terrain ids (optional)
  double* d_grid = nullptr;       // height grid of TWB_GRID_CSV (optional)
  float* d_gmap = nullptr;        // elevation layer of TWB_GRID_MAP (optional)
  double* d_XT = nullptr;         // [ld/32][n+1][32] instance-tiled iterates; row n == 0
  double* d_GT = nullptr;         // [ld/32][m][32] instance-tiled constraint values (staging of g)
  int* d_TD = nullptr;            // [ld/32] per-tile completion counters of the output kernels (zero between evaluations)
  double* d_FS = nullptr;         // [ld/32][n_dyn][6 n_ee][32] feet positions / forces per dynamic sample (optimised durations only)
  // staging for the host-pointer variant
  double *d_x = nullptr, *d_g = nullptr, *d_jac = nullptr, *d_cost = nullptr, *d_grad = nullptr;
  int* d_status = nullptr;
  cudaStream_t stream = nullptr, aux0 = nullptr, aux1 = nullptr;
  cudaStream_t s_in = nullptr, s_out = nullptr;   // copy streams of the pipelined host-pointer evaluation
  std::vector<cudaEvent_t> ev_chunk;              // per chunk: H2D done, kernels done
  int e2e_chunk = 512;                            // instances per chunk of twb_batch_eval_host (TWB_E2E_CHUNK)
  std::vector<cudaEvent_t> ev;    // fork/join events of the two-stream pipeline
  int launches_last = 0;
  cudaAccessPolicyWindow l2_window{};            // XT + GT persisting in the L2 (experiment, TWB_L2_PERSIST=1)
  bool use_l2_window = false;
  std::vector<std::pair<void*, size_t>> scratch;   // device scratch of the post-processing calls, grown on demand, freed with the batch
  // CUDA graphs of twb_batch_eval_device: one evaluation is 4 - 6 kernels on three streams joined by events; replayed as a
  // graph, the dependencies are resolved on the device instead of through cross-stream event waits.  One instantiated graph
  // per distinct argument set (a solver loop alternates between a few buffers), least recently used replaced.
  struct EvalGraph { const void* x; void *g, *jac, *cost, *grad, *status; unsigned flags; cudaGraphExec_t exec; int launches; unsigned long long used; };
  std::vector<EvalGraph> graphs;
  unsigned long long graph_clock = 0;
  twb::LmPattern lm_pat{};        // device copies of the pattern, its transpose and the bounds for twb_batch_lm_step_device (first use)
  const double *d_xl = nullptr, *d_xu = nullptr;
  bool lm_ready = false;
  int use_graphs = 1;             // TWB_GRAPH=0 disables; set to 0 when a capture fails
  // twb_batch_eval_device walks batches of 1.5 .. 3.5 x this many instances in chunks (one after the other on the same streams).
  // Measured (profiles/README.md, experiment 55; fixed durations): 8192 instances in one go cost 145.8 us per 4096 — the
  // pipeline's weakest size — against 137 us in two chunks; 16 384 and more are as fast (or faster) in one go.  0: never.
  size_t eval_chunk = 4096;
  // Sample tables of the post-processing calls (Formulation::TrajectoryTables / SampleTables), built on the host and uploaded
  // once per key: trajectory dt, the footstep plan's 0.01 s grid, or the initial-guess sample times.  Least recently used
  // replaced beyond kMaxPostTables; a CUDA graph that captured a post-processing call refers to its entry's memory.
  struct PostTables {
    int kind; std::vector<double> key;
    void* mem;                              // one device allocation holding the arrays below
    const twb::SplineSample* samples;       // [n_steps][2 + 2 n_ee]
    const double* times;                    // [n_steps]
    const int* contact;                     // fixed durations: [n_steps][n_ee] flags; optimised: in_contact_at_start [n_ee]
    const int* codes;                       // footstep plan, fixed durations: [n_codes] (step << 4) | contact mask of each change
    int n_steps, n_codes;
    unsigned long long used;
  };
  std::vector<PostTables> post_tables;
  unsigned long long post_clock = 0;
};

namespace {
// instances per chunk of twb_batch_eval_device (twb_batch::eval_chunk): the whole batch unless it is 1.5 .. 3.5 chunks long
size_t EvalChunk(const twb_batch* b) {
  const size_t B = (size_t)b->B, group = 32 * (size_t)std::max(b->plan.nc_jac, 1);
  if (!b->eval_chunk || g_prof_on || b->plan.n_phase_defs > 0) return B;
  const size_t chunk = (b->eval_chunk + group - 1) / group * group;
  return (2 * B >= 3 * chunk && 2 * B <= 7 * chunk) ? chunk : B;
}
// cached graphs hold the batch's plan and buffers by value: dropped whenever those change
void DropGraphs(twb_batch* b) {
  for (auto& gr : b->graphs) cudaGraphExecDestroy(gr.exec);
  b->graphs.clear();
}
// slot `slot` of the batch's scratch pool with at least `bytes` bytes (the post-processing entry points synchronise before
// they return and a batch has one caller at a time, so the slots are free again at the next call)
cudaError_t ScratchAlloc(twb_batch* b, int slot, void** p, size_t bytes) {
  if ((int)b->scratch.size() <= slot) b->scratch.resize(slot + 1, {nullptr, 0});
  auto& s = b->scratch[slot];
  if (s.second < bytes || !s.first) {
    cudaFree(s.first); s = {nullptr, 0};
    cudaError_t e = cudaMalloc(&s.first, std::max<size_t>(bytes, 256));
    if (e != cudaSuccess) { s.first = nullptr; return e; }
    s.second = std::max<size_t>(bytes, 256);
  }
  *p = s.first;
  return cudaSuccess;
}
enum { kPostTrajectory = 0, kPostInitialGuess = 1, kPostFootstep = 2 };
constexpr int kMaxPostTables = 8;
constexpr double kFootstepDt = 0.01;   // footstep_plan_extractor.h:87

// the cached tables of (kind, key), built and uploaded (blocking copy) on the first call with that key
int GetPostTables(twb_batch* b, int kind, const double* key, int n_key, const twb_batch::PostTables** out) {
  for (auto& t : b->post_tables)
    if (t.kind == kind && (int)t.key.size() == n_key && std::memcmp(t.key.data(), key, sizeof(double) * n_key) == 0) {
      t.used = ++b->post_clock; *out = &t; return TWB_OK;
    }
  const twb::Formulation& f = b->prob->f;
  const int n_ee = f.spec.n_ee;
  std::vector<double> times; std::vector<twb::SplineSample> samples; std::vector<int> contact, codes;
  int rc;
  if (kind == kPostInitialGuess) { times.assign(key, key + n_key); rc = f.SampleTables(times, &samples, &contact); }
  else rc = f.TrajectoryTables(key[0], &times, &samples, &contact);
  if (rc != TWB_OK) return Fail(rc, kind == kPostInitialGuess ? "bad sample times" : "bad dt");
  if (kind != kPostInitialGuess && f.optimize_timings) { contact.clear(); for (int e = 0; e < n_ee; ++e) contact.push_back(f.spec.in_contact_at_start[e] != 0); }
  if (kind == kPostFootstep && !f.optimize_timings)   // the first step and every change of the contact set (HasEndEffectorContactChanged)
    for (size_t k = 0, prev = 0; k < times.size(); ++k) {
      size_t mask = 0;
      for (int e = 0; e < n_ee; ++e) mask |= (size_t)(contact[k * n_ee + e] != 0) << e;
      if (k == 0 || mask != prev) codes.push_back((int)((k << 4) | mask));
      prev = mask;
    }
  // one allocation, every array at a 256-byte boundary
  auto up = [](size_t bytes) { return (bytes + 255) & ~(size_t)255; };
  const size_t o_times = up(sizeof(twb::SplineSample) * samples.size()), o_contact = o_times + up(sizeof(double) * times.size()),
               o_codes = o_contact + up(sizeof(int) * contact.size()), total = o_codes + up(sizeof(int) * codes.size());
  std::vector<char> host(total, 0);
  std::memcpy(host.data(), samples.data(), sizeof(twb::SplineSample) * samples.size());
  std::memcpy(host.data() + o_times, times.data(), sizeof(double) * times.size());
  std::memcpy(host.data() + o_contact, contact.data(), sizeof(int) * contact.size());
  std::memcpy(host.data() + o_codes, codes.data(), sizeof(int) * codes.size());
  if ((int)b->post_tables.size() >= kMaxPostTables) {   // replace the least recently used (cudaFree waits for the work in flight)
    size_t lru = 0;
    for (size_t i = 1; i < b->post_tables.size(); ++i) if (b->post_tables[i].used < b->post_tables[lru].used) lru = i;
    cudaFree(b->post_tables[lru].mem);
    b->post_tables.erase(b->post_tables.begin() + lru);
  }
  void* mem = nullptr;
  cudaError_t e = cudaMalloc(&mem, std::max<size_t>(total, 256));
  if (e != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = cudaMemcpy(mem, host.data(), total, cudaMemcpyHostToDevice)) != cudaSuccess) { cudaFree(mem); return CudaFail(e, "table upload"); }
  char* d = static_cast<char*>(mem);
  b->post_tables.push_back({kind, std::vector<double>(key, key + n_key), mem, reinterpret_cast<const twb::SplineSample*>(d),
                            reinterpret_cast<const double*>(d + o_times), reinterpret_cast<const int*>(d + o_contact),
                            reinterpret_cast<const int*>(d + o_codes), (int)times.size(), (int)codes.size(), ++b->post_clock});
  *out = &b->post_tables.back();
  return TWB_OK;
}

// The device cores of the post-processing calls: enqueue on `s`, device pointers only.  The _host variants copy x up, call
// these on the batch's stream, copy the results down and synchronise.
int TrajectoryCore(twb_batch* b, const double* x, double dt, double* out, cudaStream_t s) {
  const twb_batch::PostTables* t = nullptr;
  int rc = GetPostTables(b, kPostTrajectory, &dt, 1, &t);
  if (rc != TWB_OK) return rc;
  rc = twb::LaunchTrajectory(b->plan, x, b->d_XT, t->samples, t->contact, t->n_steps, out, b->B, s);
  return rc != 0 ? CudaFail(static_cast<cudaError_t>(rc), "trajectory kernel launch") : TWB_OK;
}
int InitialGuessCore(twb_batch* b, const double* x, const double* times, int n_times, double* out, cudaStream_t s) {
  const twb_batch::PostTables* t = nullptr;
  int rc = GetPostTables(b, kPostInitialGuess, times, n_times, &t);
  if (rc != TWB_OK) return rc;
  rc = twb::LaunchInitialGuess(b->plan, x, b->d_XT, t->samples, t->times, n_times, out, b->B, s);
  return rc != 0 ? CudaFail(static_cast<cudaError_t>(rc), "initial-guess kernel launch") : TWB_OK;
}
int FootstepCore(twb_batch* b, const double* x, double time_horizon, int* n_states, double* out, cudaStream_t s) {
  const twb_batch::PostTables* t = nullptr;
  const double dt = kFootstepDt;
  int rc = GetPostTables(b, kPostFootstep, &dt, 1, &t);
  if (rc != TWB_OK) return rc;
  int max_states = 0;
  twb_problem_footstep_plan_dims(b->prob, &max_states, nullptr);
  rc = twb::LaunchFootstepPlan(b->plan, x, b->d_XT, t->samples, t->times, t->contact, t->codes, t->n_codes, t->n_steps, time_horizon,
                               max_states, n_states, out, b->B, s);
  return rc != 0 ? CudaFail(static_cast<cudaError_t>(rc), "footstep-plan kernel launch") : TWB_OK;
}
int NearestPlanesCore(twb_batch* b, const double* plan, const int* n_states, const int* poly_offsets, int n_polys, const double* vertices,
                      int* contact_set, cudaStream_t s) {
  int max_states = 0;
  twb_problem_footstep_plan_dims(b->prob, &max_states, nullptr);
  const int rc = twb::LaunchNearestPlanes(plan, n_states, max_states, b->prob->f.spec.n_ee, poly_offsets, n_polys, vertices, contact_set, b->B, s);
  return rc != 0 ? CudaFail(static_cast<cudaError_t>(rc), "nearest-plane kernel launch") : TWB_OK;
}
}  // namespace

extern "C" {

const char* twb_last_error(void) { return g_err.c_str(); }
const char* twb_version(void) { return "towr_b200 0.1 (sm_100a, fp64)"; }

int twb_problem_create(const twb_spec* spec, twb_problem** out) {
  if (!spec || !out) return Fail(TWB_ERR_INVALID, "null argument");
  *out = nullptr;
  twb_problem* p = new (std::nothrow) twb_problem();
  if (!p) return Fail(TWB_ERR_INVALID, "out of memory");
  std::string err;
  int rc = TWB_OK;
  try { rc = p->f.Build(*spec, &err); } catch (const std::exception& e) { rc = TWB_ERR_INVALID; err = e.what(); }
  if (rc != TWB_OK) { delete p; return Fail(rc, err); }
  *out = p;
  return TWB_OK;
}
void twb_problem_destroy(twb_problem* p) { delete p; }

int twb_problem_dims(const twb_problem* p, int* n, int* m, int* nnz) {
  if (!p) return Fail(TWB_ERR_INVALID, "null problem");
  if (n) *n = p->f.n;
  if (m) *m = p->f.m;
  if (nnz) *nnz = p->f.nnz;
  return TWB_OK;
}
int twb_problem_structure(const twb_problem* p, int* iRow, int* jCol) {
  if (!p || !iRow || !jCol) return Fail(TWB_ERR_INVALID, "null argument");
  for (int r = 0; r < p->f.m; ++r)
    for (int k = p->f.row_ptr[r]; k < p->f.row_ptr[r + 1]; ++k) { iRow[k] = r; jCol[k] = p->f.col_idx[k]; }
  return TWB_OK;
}
int twb_problem_row_ptr(const twb_problem* p, int* row_ptr) {
  if (!p || !row_ptr) return Fail(TWB_ERR_INVALID, "null argument");
  std::memcpy(row_ptr, p->f.row_ptr.data(), sizeof(int) * (p->f.m + 1));
  return TWB_OK;
}
int twb_problem_bounds(const twb_problem* p, double* xl, double* xu, double* gl, double* gu) {
  if (!p) return Fail(TWB_ERR_INVALID, "null problem");
  if (xl) std::memcpy(xl, p->f.x_lower.data(), sizeof(double) * p->f.n);
  if (xu) std::memcpy(xu, p->f.x_upper.data(), sizeof(double) * p->f.n);
  if (gl) std::memcpy(gl, p->f.g_lower.data(), sizeof(double) * p->f.m);
  if (gu) std::memcpy(gu, p->f.g_upper.data(), sizeof(double) * p->f.m);
  return TWB_OK;
}
int twb_problem_has_cost(const twb_problem* p) { return (p && p->f.has_cost) ? 1 : 0; }

int twb_problem_x0(const twb_problem* p, double* x0) {
  if (!p || !x0) return Fail(TWB_ERR_INVALID, "null argument");
  std::memcpy(x0, p->f.x0.data(), sizeof(double) * p->f.n);
  return TWB_OK;
}
int twb_problem_goal_instances(const twb_problem* p, int n_goals, const double* goals, double* x0, double* xl, double* xu) {
  if (!p || !goals || n_goals < 0) return Fail(TWB_ERR_INVALID, "bad argument");
  const size_t n = (size_t)p->f.n;
  for (int i = 0; i < n_goals; ++i) {
    const double* gpose = goals + 6 * (size_t)i;
    int rc = p->f.GoalInstance(gpose, gpose + 3, x0 ? x0 + i * n : nullptr, xl ? xl + i * n : nullptr, xu ? xu + i * n : nullptr);
    if (rc != TWB_OK) return Fail(rc, "goal instance");
  }
  return TWB_OK;
}
int twb_layout_num_variable_sets(const twb_problem* p) { return p ? (int)p->f.var_sets.size() : 0; }
int twb_layout_num_constraint_sets(const twb_problem* p) { return p ? (int)p->f.con_sets.size() : 0; }
static int CopyComponent(const std::vector<twb::Component>& v, int i, char* name, int cap, int* start, int* count) {
  if (i < 0 || i >= (int)v.size()) return Fail(TWB_ERR_INVALID, "component index out of range");
  if (name && cap > 0) std::snprintf(name, cap, "%s", v[i].name.c_str());
  if (start) *start = v[i].start;
  if (count) *count = v[i].count;
  return TWB_OK;
}
int twb_layout_variable_set(const twb_problem* p, int i, char* name, int cap, int* col_start, int* n_cols) {
  if (!p) return Fail(TWB_ERR_INVALID, "null problem");
  return CopyComponent(p->f.var_sets, i, name, cap, col_start, n_cols);
}
int twb_layout_constraint_set(const twb_problem* p, int i, char* name, int cap, int* row_start, int* n_rows) {
  if (!p) return Fail(TWB_ERR_INVALID, "null problem");
  return CopyComponent(p->f.con_sets, i, name, cap, row_start, n_rows);
}

int twb_batch_create(const twb_problem* p, int batch_size, int device, twb_batch** out) {
  if (!p || !out || batch_size <= 0) return Fail(TWB_ERR_INVALID, "bad argument");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return Fail(TWB_ERR_NO_DEVICE, "no CUDA device: towr_b200 has no CPU evaluation path");
  if (device < 0 || device >= count) return Fail(TWB_ERR_INVALID, "device index out of range");
  if ((e = cudaSetDevice(device)) != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  twb_batch* b = new (std::nothrow) twb_batch();
  if (!b) return Fail(TWB_ERR_INVALID, "out of memory");
  b->prob = p; b->B = batch_size; b->device = device;
  const twb::HostTables& t = p->f.tables;
  b->plan = t.plan;
#define TWB_UP(field)                                                                  \
  if ((e = Upload(t.field, &b->plan.field, &b->owned)) != cudaSuccess) {               \
    twb_batch_destroy(b);                                                              \
    return CudaFail(e, "table upload");                                                \
  }
  TWB_UP(samples) TWB_UP(dyn) TWB_UP(rom) TWB_UP(groups) TWB_UP(terr) TWB_UP(force) TWB_UP(swing) TWB_UP(acc)
  TWB_UP(base_motion) TWB_UP(cost) TWB_UP(pairs) TWB_UP(coefs) TWB_UP(cta_lists) TWB_UP(dyn_ang_basis)
  TWB_UP(phase_defs) TWB_UP(phase_polys) TWB_UP(phase_units) TWB_UP(exts) TWB_UP(goal_vars) TWB_UP(const_runs) TWB_UP(const_vals)
#undef TWB_UP
  if (std::getenv("TWB_PROFILE") && !g_prof_on) { g_prof_on = true; twb::g_after_launch = ProfHook; std::atexit(ProfReport); }
  if (g_prof_on) std::fprintf(stderr, "[twb profile] n=%d m=%d nnz=%d\n", b->plan.n, b->plan.m, b->plan.nnz);
  if (const char* v = std::getenv("TWB_E2E_CHUNK")) b->e2e_chunk = std::max(32, std::atoi(v));
  if (const char* v = std::getenv("TWB_GRAPH")) b->use_graphs = std::atoi(v) != 0;
  if (const char* v = std::getenv("TWB_EVAL_CHUNK")) b->eval_chunk = (size_t)std::max(0, std::atoi(v));
  // whole groups of nc interleaved tiles (kernels.cu: TileInstance); nc = 1 unless the Jacobian row length is not a multiple of 4
  const size_t group = 32 * (size_t)std::max(b->plan.nc_jac, 1);
  b->ld = ((size_t)batch_size + group - 1) / group * group;
  const size_t xt_bytes = (size_t)(b->plan.n + 1) * b->ld * sizeof(double);
  // XT and GT live in ONE allocation, so that one L2 access-policy window can cover both staging matrices (TWB_L2_PERSIST=1;
  // measured, profiles/README.md experiment 39: marking them persisting makes the step SLOWER, 175 instead of 139 us — off)
  const size_t xt_padded = (xt_bytes + 255) & ~(size_t)255, gt_bytes = (size_t)std::max(b->plan.m, 1) * b->ld * sizeof(double);
  if ((e = cudaMalloc(reinterpret_cast<void**>(&b->d_XT), xt_padded + gt_bytes)) != cudaSuccess ||
      (e = cudaMemset(b->d_XT, 0, xt_bytes)) != cudaSuccess) {
    twb_batch_destroy(b);
    return CudaFail(e, "state allocation");
  }
  b->d_GT = reinterpret_cast<double*>(reinterpret_cast<char*>(b->d_XT) + xt_padded);
  if ((e = cudaMalloc(reinterpret_cast<void**>(&b->d_TD), sizeof(int) * (b->ld / 32))) != cudaSuccess ||
      (e = cudaMemset(b->d_TD, 0, sizeof(int) * (b->ld / 32))) != cudaSuccess) {
    twb_batch_destroy(b);
    return CudaFail(e, "state allocation");
  }
  if (b->plan.n_phase_defs > 0 && b->plan.n_dyn > 0 &&
      (e = cudaMalloc(reinterpret_cast<void**>(&b->d_FS), (size_t)b->plan.n_dyn * 6 * b->plan.n_ee * b->ld * sizeof(double))) != cudaSuccess) {
    twb_batch_destroy(b);
    return CudaFail(e, "state allocation");
  }
  {
    const char* v = std::getenv("TWB_L2_PERSIST");
    cudaDeviceProp prop{};
    if (v && std::atoi(v) != 0 && cudaGetDeviceProperties(&prop, device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
      const size_t want = xt_padded + gt_bytes, cap = (size_t)prop.persistingL2CacheMaxSize;
      size_t cur = 0; cudaDeviceGetLimit(&cur, cudaLimitPersistingL2CacheSize);
      if (cur < std::min(want, cap)) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, std::min(want, cap));
      b->l2_window.base_ptr = b->d_XT;
      b->l2_window.num_bytes = std::min(want, (size_t)prop.accessPolicyMaxWindowSize);
      b->l2_window.hitRatio = want <= cap ? 1.0f : (float)((double)cap / (double)want);
      b->l2_window.hitProp = cudaAccessPropertyPersisting;
      b->l2_window.missProp = cudaAccessPropertyNormal;
      b->use_l2_window = true;
    }
  }
  if ((e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&b->aux0, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&b->aux1, cudaStreamNonBlocking)) != cudaSuccess) {
    twb_batch_destroy(b);
    return CudaFail(e, "cudaStreamCreate");
  }
  b->ev.assign(3, nullptr);
  for (auto& ev : b->ev)
    if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) {
      twb_batch_destroy(b);
      return CudaFail(e, "cudaEventCreate");
    }
  *out = b;
  return TWB_OK;
}

void twb_batch_destroy(twb_batch* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  DropGraphs(b);
  if (b->use_l2_window) cudaCtxResetPersistingL2Cache();   // lines of XT / GT must not stay pinned in the L2 after the batch is gone
  for (void* p : b->owned) cudaFree(p);
  for (auto& sc : b->scratch) cudaFree(sc.first);
  for (auto& t : b->post_tables) cudaFree(t.mem);
  cudaFree(b->d_terrain); cudaFree(b->d_grid); cudaFree(b->d_gmap); cudaFree(b->d_XT); cudaFree(b->d_FS); cudaFree(b->d_TD);   // (d_GT is part of d_XT's allocation)
  for (auto ev : b->ev) if (ev) cudaEventDestroy(ev);
  if (b->aux0) cudaStreamDestroy(b->aux0);
  if (b->aux1) cudaStreamDestroy(b->aux1);
  if (b->s_in) cudaStreamDestroy(b->s_in);
  if (b->s_out) cudaStreamDestroy(b->s_out);
  for (auto ev : b->ev_chunk) cudaEventDestroy(ev);
  cudaFree(b->d_x); cudaFree(b->d_g); cudaFree(b->d_jac); cudaFree(b->d_cost); cudaFree(b->d_grad); cudaFree(b->d_status);
  if (b->stream) cudaStreamDestroy(b->stream);
  delete b;
}

int twb_batch_set_terrains(twb_batch* b, const int* terrain_ids) {
  if (!b) return Fail(TWB_ERR_INVALID, "null batch");
  cudaSetDevice(b->device);
  DropGraphs(b);
  if (!terrain_ids) { cudaFree(b->d_terrain); b->d_terrain = nullptr; return TWB_OK; }
  for (int i = 0; i < b->B; ++i)
    if (terrain_ids[i] < 0 || terrain_ids[i] > TWB_GRID_MAP) return Fail(TWB_ERR_INVALID, "unknown terrain id");
  cudaError_t e;
  if (!b->d_terrain && (e = cudaMalloc(&b->d_terrain, sizeof(int) * b->B)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = cudaMemcpy(b->d_terrain, terrain_ids, sizeof(int) * b->B, cudaMemcpyHostToDevice)) != cudaSuccess)
    return CudaFail(e, "cudaMemcpy");
  return TWB_OK;
}

int twb_batch_set_grid_terrain(twb_batch* b, const double* heights, int rows, int cols) {
  if (!b) return Fail(TWB_ERR_INVALID, "null batch");
  cudaSetDevice(b->device);
  DropGraphs(b);
  cudaFree(b->d_grid); b->d_grid = nullptr;
  b->plan.grid = nullptr; b->plan.grid_rows = b->plan.grid_cols = 0;
  if (!heights) return TWB_OK;
  if (rows <= 0 || cols <= 0 || (long long)rows * cols > (1ll << 28)) return Fail(TWB_ERR_INVALID, "bad grid size");
  cudaError_t e;
  const size_t bytes = sizeof(double) * (size_t)rows * cols;
  if ((e = cudaMalloc(reinterpret_cast<void**>(&b->d_grid), bytes)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = cudaMemcpy(b->d_grid, heights, bytes, cudaMemcpyHostToDevice)) != cudaSuccess) return CudaFail(e, "cudaMemcpy");
  b->plan.grid = b->d_grid; b->plan.grid_rows = rows; b->plan.grid_cols = cols;
  return TWB_OK;
}

int twb_batch_set_grid_map(twb_batch* b, const float* heights, int size_x, int size_y, double resolution, double pos_x, double pos_y) {
  if (!b) return Fail(TWB_ERR_INVALID, "null batch");
  cudaSetDevice(b->device);
  DropGraphs(b);
  cudaFree(b->d_gmap); b->d_gmap = nullptr;
  b->plan.gmap = nullptr; b->plan.gmap_sx = b->plan.gmap_sy = 0; b->plan.gmap_res = 1.0; b->plan.gmap_px = b->plan.gmap_py = 0.0;
  if (!heights) return TWB_OK;
  if (size_x <= 0 || size_y <= 0 || (long long)size_x * size_y > (1ll << 28) || !(resolution > 0.0) || !std::isfinite(resolution) ||
      !std::isfinite(pos_x) || !std::isfinite(pos_y))
    return Fail(TWB_ERR_INVALID, "bad grid map geometry");
  cudaError_t e;
  const size_t bytes = sizeof(float) * (size_t)size_x * size_y;
  if ((e = cudaMalloc(reinterpret_cast<void**>(&b->d_gmap), bytes)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = cudaMemcpy(b->d_gmap, heights, bytes, cudaMemcpyHostToDevice)) != cudaSuccess) return CudaFail(e, "cudaMemcpy");
  b->plan.gmap = b->d_gmap; b->plan.gmap_sx = size_x; b->plan.gmap_sy = size_y; b->plan.gmap_res = resolution; b->plan.gmap_px = pos_x; b->plan.gmap_py = pos_y;
  return TWB_OK;
}

int twb_batch_goal_instances_device(twb_batch* b, const double* goals, double* x0, double* x_lower, double* x_upper, void* stream) {
  if (!b || !goals) return Fail(TWB_ERR_INVALID, "null argument");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb::Formulation& f = b->prob->f;
  int rc = twb::LaunchGoalInstances(b->plan, f.tables.goal_setup, goals, b->d_terrain, f.spec.terrain, x0, x_lower, x_upper, b->B, static_cast<cudaStream_t>(stream));
  if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "goal-instance kernel launch");
  return TWB_OK;
}

int twb_problem_trajectory_dims(const twb_problem* p, double dt, int* n_samples, int* n_values) {
  if (!p) return Fail(TWB_ERR_INVALID, "null problem");
  std::vector<double> times; std::vector<twb::SplineSample> samples; std::vector<int> contact;
  int rc = p->f.TrajectoryTables(dt, &times, &samples, &contact);
  if (rc != TWB_OK) return Fail(rc, "bad dt");
  if (n_samples) *n_samples = (int)times.size();
  if (n_values) *n_values = 19 + 13 * p->f.spec.n_ee;
  return TWB_OK;
}

int twb_batch_sample_trajectory_host(twb_batch* b, const double* x, double dt, double* out) {
  if (!b || !x || !out) return Fail(TWB_ERR_INVALID, "null argument");
  if (!(dt > 0.0)) return Fail(TWB_ERR_INVALID, "bad dt");
  const twb::Formulation& f = b->prob->f;
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb_batch::PostTables* t = nullptr;
  int rc = GetPostTables(b, kPostTrajectory, &dt, 1, &t);
  if (rc != TWB_OK) return rc;
  const size_t B = b->B, K = 19 + 13 * (size_t)f.spec.n_ee, n_steps = t->n_steps;
  double* d_out = nullptr;   // scratch buffers stay with the batch (twb_batch::scratch) and are reused by the next call
  if (!b->d_x && (e = cudaMalloc(reinterpret_cast<void**>(&b->d_x), sizeof(double) * B * f.n)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = ScratchAlloc(b, 0, reinterpret_cast<void**>(&d_out), sizeof(double) * B * n_steps * K)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  cudaStream_t s = b->stream;
  cudaMemcpyAsync(b->d_x, x, sizeof(double) * B * f.n, cudaMemcpyHostToDevice, s);
  rc = TrajectoryCore(b, b->d_x, dt, d_out, s);
  if (rc == TWB_OK) cudaMemcpyAsync(out, d_out, sizeof(double) * B * n_steps * K, cudaMemcpyDeviceToHost, s);
  e = cudaStreamSynchronize(s);
  if (rc != TWB_OK) return rc;
  if (e != cudaSuccess) return CudaFail(e, "trajectory sampling");
  return TWB_OK;
}

int twb_batch_sample_trajectory_device(twb_batch* b, const double* x, double dt, double* out, void* stream) {
  if (!b || !x || !out) return Fail(TWB_ERR_INVALID, "null argument");
  if (!(dt > 0.0)) return Fail(TWB_ERR_INVALID, "bad dt");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  return TrajectoryCore(b, x, dt, out, static_cast<cudaStream_t>(stream));
}

int twb_batch_initial_guess_host(twb_batch* b, const double* x, const double* times, int n_times, double* out) {
  if (!b || !x || !times || !out || n_times <= 0) return Fail(TWB_ERR_INVALID, "null argument");
  const twb::Formulation& f = b->prob->f;
  if (f.spec.n_ee > 4) return Fail(TWB_ERR_UNSUPPORTED, "the initial-guess layout holds at most 4 feet");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const size_t B = b->B;
  double* d_out = nullptr;   // scratch buffers stay with the batch (twb_batch::scratch) and are reused by the next call
  if (!b->d_x && (e = cudaMalloc(reinterpret_cast<void**>(&b->d_x), sizeof(double) * B * f.n)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = ScratchAlloc(b, 0, reinterpret_cast<void**>(&d_out), sizeof(double) * B * n_times * 49)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  cudaStream_t s = b->stream;
  cudaMemcpyAsync(b->d_x, x, sizeof(double) * B * f.n, cudaMemcpyHostToDevice, s);
  int rc = InitialGuessCore(b, b->d_x, times, n_times, d_out, s);
  if (rc == TWB_OK) cudaMemcpyAsync(out, d_out, sizeof(double) * B * n_times * 49, cudaMemcpyDeviceToHost, s);
  e = cudaStreamSynchronize(s);
  if (rc != TWB_OK) return rc;
  if (e != cudaSuccess) return CudaFail(e, "initial-guess sampling");
  return TWB_OK;
}

int twb_batch_initial_guess_device(twb_batch* b, const double* x, const double* times, int n_times, double* out, void* stream) {
  if (!b || !x || !times || !out || n_times <= 0) return Fail(TWB_ERR_INVALID, "null argument");
  if (b->prob->f.spec.n_ee > 4) return Fail(TWB_ERR_UNSUPPORTED, "the initial-guess layout holds at most 4 feet");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  return InitialGuessCore(b, x, times, n_times, out, static_cast<cudaStream_t>(stream));
}

int twb_problem_footstep_plan_dims(const twb_problem* p, int* max_states, int* n_values) {
  if (!p) return Fail(TWB_ERR_INVALID, "null problem");
  int changes = 0;
  for (int e = 0; e < p->f.spec.n_ee; ++e) changes += p->f.spec.n_phases[e] - 1;
  if (max_states) *max_states = 1 + changes;   // the first state + at most one footstep state per phase change of a foot
  if (n_values) *n_values = 2 + 4 * p->f.spec.n_ee;
  return TWB_OK;
}

int twb_batch_footstep_plan_host(twb_batch* b, const double* x, double time_horizon, int* n_states, double* out) {
  if (!b || !x || !n_states || !out) return Fail(TWB_ERR_INVALID, "null argument");
  const twb::Formulation& f = b->prob->f;
  int max_states = 0, V = 0;
  twb_problem_footstep_plan_dims(b->prob, &max_states, &V);
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const size_t B = b->B;
  double* d_out = nullptr; int* d_count = nullptr;   // scratch buffers stay with the batch (twb_batch::scratch) and are reused by the next call
  if (!b->d_x && (e = cudaMalloc(reinterpret_cast<void**>(&b->d_x), sizeof(double) * B * f.n)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = ScratchAlloc(b, 0, reinterpret_cast<void**>(&d_out), sizeof(double) * B * max_states * V)) != cudaSuccess ||
      (e = ScratchAlloc(b, 1, reinterpret_cast<void**>(&d_count), sizeof(int) * B)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  cudaStream_t s = b->stream;
  cudaMemcpyAsync(b->d_x, x, sizeof(double) * B * f.n, cudaMemcpyHostToDevice, s);
  int rc = FootstepCore(b, b->d_x, time_horizon, d_count, d_out, s);
  if (rc == TWB_OK) {
    cudaMemcpyAsync(out, d_out, sizeof(double) * B * max_states * V, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(n_states, d_count, sizeof(int) * B, cudaMemcpyDeviceToHost, s);
  }
  e = cudaStreamSynchronize(s);
  if (rc != TWB_OK) return rc;
  if (e != cudaSuccess) return CudaFail(e, "footstep-plan extraction");
  return TWB_OK;
}

int twb_batch_footstep_plan_device(twb_batch* b, const double* x, double time_horizon, int* n_states, double* out, void* stream) {
  if (!b || !x || !n_states || !out) return Fail(TWB_ERR_INVALID, "null argument");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  return FootstepCore(b, x, time_horizon, n_states, out, static_cast<cudaStream_t>(stream));
}

int twb_batch_nearest_planes_host(twb_batch* b, const double* plan, const int* n_states, const int* poly_offsets, int n_polys,
                                  const double* vertices, int* contact_set) {
  if (!b || !plan || !n_states || !poly_offsets || !contact_set || n_polys < 0 || (n_polys > 0 && !vertices)) return Fail(TWB_ERR_INVALID, "null argument");
  for (int k = 0; k < n_polys; ++k) if (poly_offsets[k + 1] < poly_offsets[k] || poly_offsets[k] < 0) return Fail(TWB_ERR_INVALID, "polygon offsets must ascend");
  int max_states = 0, V = 0;
  twb_problem_footstep_plan_dims(b->prob, &max_states, &V);
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const size_t B = b->B, n_ee = b->prob->f.spec.n_ee, n_vert = n_polys > 0 ? (size_t)poly_offsets[n_polys] : 0;
  double* d_plan = nullptr; int* d_count = nullptr; int* d_off = nullptr; double* d_vert = nullptr; int* d_out = nullptr;
  // scratch buffers stay with the batch (twb_batch::scratch) and are reused by the next call
  if ((e = ScratchAlloc(b, 0, reinterpret_cast<void**>(&d_plan), sizeof(double) * B * max_states * V)) != cudaSuccess ||
      (e = ScratchAlloc(b, 1, reinterpret_cast<void**>(&d_count), sizeof(int) * B)) != cudaSuccess ||
      (e = ScratchAlloc(b, 2, reinterpret_cast<void**>(&d_off), sizeof(int) * (n_polys + 1))) != cudaSuccess ||
      (e = ScratchAlloc(b, 3, reinterpret_cast<void**>(&d_vert), sizeof(double) * 2 * std::max<size_t>(n_vert, 1))) != cudaSuccess ||
      (e = ScratchAlloc(b, 4, reinterpret_cast<void**>(&d_out), sizeof(int) * B * max_states * n_ee)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  cudaStream_t s = b->stream;
  cudaMemcpyAsync(d_plan, plan, sizeof(double) * B * max_states * V, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(d_count, n_states, sizeof(int) * B, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(d_off, poly_offsets, sizeof(int) * (n_polys + 1), cudaMemcpyHostToDevice, s);
  if (n_vert) cudaMemcpyAsync(d_vert, vertices, sizeof(double) * 2 * n_vert, cudaMemcpyHostToDevice, s);
  int rc = NearestPlanesCore(b, d_plan, d_count, d_off, n_polys, d_vert, d_out, s);
  if (rc == TWB_OK) cudaMemcpyAsync(contact_set, d_out, sizeof(int) * B * max_states * n_ee, cudaMemcpyDeviceToHost, s);
  e = cudaStreamSynchronize(s);
  if (rc != TWB_OK) return rc;
  if (e != cudaSuccess) return CudaFail(e, "nearest-plane lookup");
  return TWB_OK;
}

int twb_batch_nearest_planes_device(twb_batch* b, const double* plan, const int* n_states, const int* poly_offsets, int n_polys,
                                    const double* vertices, int* contact_set, void* stream) {
  if (!b || !plan || !n_states || !poly_offsets || !contact_set || n_polys < 0 || (n_polys > 0 && !vertices)) return Fail(TWB_ERR_INVALID, "null argument");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  return NearestPlanesCore(b, plan, n_states, poly_offsets, n_polys, vertices, contact_set, static_cast<cudaStream_t>(stream));
}

int twb_batch_linear_equality_host(twb_batch* b, const double* x, int var_set, const double* M, int rows, double* g) {
  if (!b || !x || !M || !g || rows <= 0) return Fail(TWB_ERR_INVALID, "bad argument");
  const twb::Formulation& f = b->prob->f;
  if (var_set < 0 || var_set >= (int)f.var_sets.size()) return Fail(TWB_ERR_INVALID, "variable set index out of range");
  const int col0 = f.var_sets[var_set].start, n_cols = f.var_sets[var_set].count;
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const size_t B = b->B;
  double* d_M = nullptr; double* d_g = nullptr;
  auto cleanup = [] {};   // scratch buffers stay with the batch (twb_batch::scratch) and are reused by the next call
  if (!b->d_x && (e = cudaMalloc(reinterpret_cast<void**>(&b->d_x), sizeof(double) * B * f.n)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = ScratchAlloc(b, 0, reinterpret_cast<void**>(&d_M), sizeof(double) * (size_t)rows * n_cols)) != cudaSuccess ||
      (e = ScratchAlloc(b, 1, reinterpret_cast<void**>(&d_g), sizeof(double) * B * rows)) != cudaSuccess) { cleanup(); return CudaFail(e, "cudaMalloc"); }
  cudaStream_t s = b->stream;
  cudaMemcpyAsync(d_M, M, sizeof(double) * (size_t)rows * n_cols, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(b->d_x, x, sizeof(double) * B * f.n, cudaMemcpyHostToDevice, s);
  int rc = twb::LaunchLinearEquality(b->plan, b->d_x, b->d_XT, col0, n_cols, d_M, rows, d_g, b->B, s);
  if (rc == 0) cudaMemcpyAsync(g, d_g, sizeof(double) * B * rows, cudaMemcpyDeviceToHost, s);
  e = cudaStreamSynchronize(s);
  cleanup();
  if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "linear-equality kernel launch");
  if (e != cudaSuccess) return CudaFail(e, "linear equality constraint");
  return TWB_OK;
}

int twb_batch_soft_constraint_host(twb_batch* b, int constraint_set, const double* weights, double* cost, double* grad) {
  if (!b || !cost || !grad) return Fail(TWB_ERR_INVALID, "null argument");
  const twb::Formulation& f = b->prob->f;
  if (constraint_set < 0 || constraint_set >= (int)f.con_sets.size()) return Fail(TWB_ERR_INVALID, "constraint set index out of range");
  if (!b->d_g || !b->d_jac) return Fail(TWB_ERR_INVALID, "no evaluation on the device yet: call twb_batch_eval_host(TWB_EVAL_G | TWB_EVAL_JAC) first");
  const int row0 = f.con_sets[constraint_set].start, n_rows = f.con_sets[constraint_set].count;
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  std::vector<double> b_avg(n_rows), w(n_rows, 1.0);
  for (int i = 0; i < n_rows; ++i) b_avg[i] = (f.g_upper[row0 + i] + f.g_lower[row0 + i]) / 2.;   // soft_constraint.cc:41-46
  if (weights) w.assign(weights, weights + n_rows);
  const size_t B = b->B;
  double *d_b = nullptr, *d_w = nullptr, *d_cost = nullptr, *d_grad = nullptr; int *d_rp = nullptr, *d_ci = nullptr;
  auto cleanup = [] {};   // scratch buffers stay with the batch (twb_batch::scratch) and are reused by the next call
  if ((e = ScratchAlloc(b, 0, reinterpret_cast<void**>(&d_b), sizeof(double) * std::max(n_rows, 1))) != cudaSuccess ||
      (e = ScratchAlloc(b, 1, reinterpret_cast<void**>(&d_w), sizeof(double) * std::max(n_rows, 1))) != cudaSuccess ||
      (e = ScratchAlloc(b, 2, reinterpret_cast<void**>(&d_cost), sizeof(double) * B)) != cudaSuccess ||
      (e = ScratchAlloc(b, 3, reinterpret_cast<void**>(&d_grad), sizeof(double) * B * f.n)) != cudaSuccess ||
      (e = ScratchAlloc(b, 4, reinterpret_cast<void**>(&d_rp), sizeof(int) * (f.m + 1))) != cudaSuccess ||
      (e = ScratchAlloc(b, 5, reinterpret_cast<void**>(&d_ci), sizeof(int) * std::max(f.nnz, 1))) != cudaSuccess) { cleanup(); return CudaFail(e, "cudaMalloc"); }
  cudaStream_t s = b->stream;
  cudaMemcpyAsync(d_b, b_avg.data(), sizeof(double) * n_rows, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(d_w, w.data(), sizeof(double) * n_rows, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(d_rp, f.row_ptr.data(), sizeof(int) * (f.m + 1), cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(d_ci, f.col_idx.data(), sizeof(int) * f.nnz, cudaMemcpyHostToDevice, s);
  int rc = twb::LaunchSoftConstraint(b->plan, b->d_g, b->d_jac, d_rp, d_ci, row0, n_rows, d_b, d_w, d_cost, d_grad, b->B, s);
  if (rc == 0) {
    cudaMemcpyAsync(cost, d_cost, sizeof(double) * B, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(grad, d_grad, sizeof(double) * B * f.n, cudaMemcpyDeviceToHost, s);
  }
  e = cudaStreamSynchronize(s);   // (pageable vectors b_avg / w stay alive until here)
  cleanup();
  if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "soft-constraint kernel launch");
  if (e != cudaSuccess) return CudaFail(e, "soft constraint");
  return TWB_OK;
}

int twb_batch_launches_per_eval(const twb_batch* b, unsigned flags) {
  if (!b) return 0;
  const twb::Plan& p = b->plan;
  const bool want_cost = b->prob->f.has_cost && (flags & TWB_EVAL_COST);
  int n = 1;   // TransposeIn
  if (flags & (TWB_EVAL_G | TWB_EVAL_JAC)) n += twb::OutKernelsPerEval(p, flags);   // DynOut [+ DynTailOut] + RomNodeOut (or RomOut, NodeOut)
  if ((flags & (TWB_EVAL_G | TWB_EVAL_JAC)) && p.n_phase_units > 0) n += 1;   // PhaseJac
  if (flags & TWB_EVAL_G) n += twb::TransposeOutPerEval(p);   // TransposeOut (not with fixed durations: the values are written directly)
  if (want_cost) n += 1;
  {   // large batches are evaluated chunk after chunk (twb_batch::eval_chunk)
    const size_t B = (size_t)b->B, chunk = EvalChunk(b);
    n *= (int)((B + chunk - 1) / chunk);
  }
  return n;
}

int twb_batch_eval_device(twb_batch* b, const double* x, double* g, double* jac, double* cost, double* grad,
                          int* status, unsigned flags, void* stream) {
  if (!b || !x) return Fail(TWB_ERR_INVALID, "null argument");
  if ((flags & TWB_EVAL_G) && !g) return Fail(TWB_ERR_INVALID, "g requested but NULL");
  if ((flags & TWB_EVAL_JAC) && !jac) return Fail(TWB_ERR_INVALID, "jac requested but NULL");
  if ((flags & TWB_EVAL_JAC) && (reinterpret_cast<uintptr_t>(jac) % 16) != 0)
    return Fail(TWB_ERR_INVALID, "jac must be 16-byte aligned (the kernels write it with 16-byte stores and TMA bulk copies)");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb::Formulation& f = b->prob->f;
  unsigned kflags = flags & (TWB_EVAL_G | TWB_EVAL_JAC);
  if (f.has_cost && (flags & TWB_EVAL_COST)) kflags |= TWB_EVAL_COST;
  int launches = 0;
  twb::SetL2Window(b->use_l2_window ? &b->l2_window : nullptr);
  // the whole batch, or chunk after chunk (twb_batch::eval_chunk), enqueued on s0 and the batch's two auxiliary streams
  auto enqueue = [&](cudaStream_t s0) -> int {
    const size_t B = (size_t)b->B;
    const size_t chunk = EvalChunk(b);
    const size_t n = f.n, m = f.m;
    for (size_t off = 0; off < B; off += chunk) {
      const size_t nb = std::min(chunk, B - off), t0 = off / 32;
      const int rc = twb::LaunchEval(b->plan, x + off * n, b->d_XT + t0 * (n + 1) * 32, b->d_GT + t0 * (size_t)std::max(f.m, 1) * 32,
                                     b->d_FS ? b->d_FS + t0 * (size_t)b->plan.n_dyn * 6 * b->plan.n_ee * 32 : nullptr, b->d_TD + t0,
                                     g ? g + off * m : nullptr, jac ? jac + off * (size_t)f.nnz : nullptr, cost ? cost + off : nullptr,
                                     grad ? grad + off * n : nullptr, status ? status + off : nullptr,
                                     b->d_terrain ? b->d_terrain + off : nullptr, f.spec.terrain, (int)nb, kflags, s0, b->aux0, b->aux1, b->ev.data(), &launches);
      if (rc != 0) return rc;
    }
    return 0;
  };
  if (b->use_graphs && !g_prof_on) {
    // replay (or first capture on the batch's own stream) the evaluation of this argument set as a CUDA graph
    twb_batch::EvalGraph* hit = nullptr;
    for (auto& gr : b->graphs)
      if (gr.x == x && gr.g == g && gr.jac == jac && gr.cost == cost && gr.grad == grad && gr.status == status && gr.flags == kflags) { hit = &gr; break; }
    if (!hit) {
      cudaGraph_t graph = nullptr; cudaGraphExec_t exec = nullptr;
      bool ok = cudaStreamBeginCapture(b->stream, cudaStreamCaptureModeRelaxed) == cudaSuccess;
      if (ok) {
        const int rc = enqueue(b->stream);
        ok = cudaStreamEndCapture(b->stream, &graph) == cudaSuccess && rc == 0 && graph != nullptr;
      }
      ok = ok && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
      if (graph) cudaGraphDestroy(graph);
      if (!ok) { cudaGetLastError(); b->use_graphs = 0; launches = 0; }   // plain launches from now on
      else {
        if (b->graphs.size() >= 16) {   // replace the least recently used
          size_t lru = 0;
          for (size_t i = 1; i < b->graphs.size(); ++i) if (b->graphs[i].used < b->graphs[lru].used) lru = i;
          cudaGraphExecDestroy(b->graphs[lru].exec);
          b->graphs.erase(b->graphs.begin() + lru);
        }
        b->graphs.push_back({x, g, jac, cost, grad, status, kflags, exec, launches, 0});
        hit = &b->graphs.back();
      }
    }
    if (hit) {
      hit->used = ++b->graph_clock;
      if ((e = cudaGraphLaunch(hit->exec, static_cast<cudaStream_t>(stream))) != cudaSuccess) return CudaFail(e, "cudaGraphLaunch");
      b->launches_last = hit->launches;
      return TWB_OK;
    }
  }
  int rc = enqueue(static_cast<cudaStream_t>(stream));
  if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "kernel launch");
  b->launches_last = launches;
  return TWB_OK;
}

int twb_batch_lm_step_device(twb_batch* b, double* x, const double* g, const double* jac, const double* x_lower, const double* x_upper,
                             double mu, double cap, int cg_iters, double* violation, void* stream) {
  if (!b || !x || !g || !jac) return Fail(TWB_ERR_INVALID, "null argument");
  if ((x_lower == nullptr) != (x_upper == nullptr)) return Fail(TWB_ERR_INVALID, "x_lower and x_upper: both or neither");
  if (!(mu >= 0.0) || !(cap > 0.0) || cg_iters < 0 || cg_iters > 10000) return Fail(TWB_ERR_INVALID, "bad solver parameter");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb::Formulation& f = b->prob->f;
  if (twb::LmSharedBytes(f.n, f.m) > 200 * 1024) return Fail(TWB_ERR_UNSUPPORTED, "problem too large for the shared-memory solver step");
  if (!b->lm_ready) {   // the pattern's transpose: entries of column j in ascending row order (what a stable sort by column yields)
    std::vector<int> col_ptr(f.n + 1, 0), slot_t(f.nnz), row_t(f.nnz);
    for (int k = 0; k < f.nnz; ++k) col_ptr[f.col_idx[k] + 1]++;
    for (int j = 0; j < f.n; ++j) col_ptr[j + 1] += col_ptr[j];
    std::vector<int> fill(col_ptr.begin(), col_ptr.end() - 1);
    for (int r = 0; r < f.m; ++r)
      for (int k = f.row_ptr[r]; k < f.row_ptr[r + 1]; ++k) { const int at = fill[f.col_idx[k]]++; slot_t[at] = k; row_t[at] = r; }
    if ((e = Upload(f.row_ptr, &b->lm_pat.row_ptr, &b->owned)) != cudaSuccess || (e = Upload(f.col_idx, &b->lm_pat.col_idx, &b->owned)) != cudaSuccess ||
        (e = Upload(col_ptr, &b->lm_pat.col_ptr, &b->owned)) != cudaSuccess || (e = Upload(slot_t, &b->lm_pat.slot_t, &b->owned)) != cudaSuccess ||
        (e = Upload(row_t, &b->lm_pat.row_t, &b->owned)) != cudaSuccess || (e = Upload(f.g_lower, &b->lm_pat.g_lower, &b->owned)) != cudaSuccess ||
        (e = Upload(f.g_upper, &b->lm_pat.g_upper, &b->owned)) != cudaSuccess || (e = Upload(f.x_lower, &b->d_xl, &b->owned)) != cudaSuccess ||
        (e = Upload(f.x_upper, &b->d_xu, &b->owned)) != cudaSuccess)
      return CudaFail(e, "pattern upload");
    {   // rows / columns in descending length (stable: ties keep their index order)
      std::vector<int> ro(f.m), co(f.n);
      for (int i = 0; i < f.m; ++i) ro[i] = i;
      for (int j = 0; j < f.n; ++j) co[j] = j;
      std::stable_sort(ro.begin(), ro.end(), [&](int a, int c) { return f.row_ptr[a + 1] - f.row_ptr[a] > f.row_ptr[c + 1] - f.row_ptr[c]; });
      std::stable_sort(co.begin(), co.end(), [&](int a, int c) { return col_ptr[a + 1] - col_ptr[a] > col_ptr[c + 1] - col_ptr[c]; });
      if ((e = Upload(ro, &b->lm_pat.row_order, &b->owned)) != cudaSuccess || (e = Upload(co, &b->lm_pat.col_order, &b->owned)) != cudaSuccess)
        return CudaFail(e, "pattern upload");
    }
    if (f.n < 65536 && f.m < 65536 && f.nnz < 65536) {
      std::vector<uint16_t> c16(f.col_idx.begin(), f.col_idx.end()), s16(slot_t.begin(), slot_t.end()), r16(row_t.begin(), row_t.end());
      if ((e = Upload(c16, &b->lm_pat.col_idx16, &b->owned)) != cudaSuccess || (e = Upload(s16, &b->lm_pat.slot_t16, &b->owned)) != cudaSuccess ||
          (e = Upload(r16, &b->lm_pat.row_t16, &b->owned)) != cudaSuccess)
        return CudaFail(e, "pattern upload");
    }
    b->lm_ready = true;
  }
  const bool own = x_lower != nullptr;
  int rc = twb::LaunchLmStep(b->lm_pat, f.n, f.m, f.nnz, x, g, jac, own ? x_lower : b->d_xl, own ? x_upper : b->d_xu, own ? (size_t)f.n : 0, mu, cap,
                             cg_iters, violation, b->B, static_cast<cudaStream_t>(stream));
  if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "solver step launch");
  return TWB_OK;
}

int twb_batch_eval_host(twb_batch* b, const double* x, double* g, double* jac, double* cost, double* grad,
                        int* status, unsigned flags) {
  if (!b || !x) return Fail(TWB_ERR_INVALID, "null argument");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb::Formulation& f = b->prob->f;
  const size_t B = b->B;
  const bool has_cost = f.has_cost && (flags & TWB_EVAL_COST);
#define TWB_ENSURE(ptr, count, T)                                                                             \
  if (!(ptr) && (e = cudaMalloc(reinterpret_cast<void**>(&(ptr)), sizeof(T) * (count))) != cudaSuccess)       \
    return CudaFail(e, "cudaMalloc");
  TWB_ENSURE(b->d_x, B * f.n, double)
  TWB_ENSURE(b->d_status, B, int)
  if (flags & TWB_EVAL_G) TWB_ENSURE(b->d_g, B * f.m, double)
  if (flags & TWB_EVAL_JAC) TWB_ENSURE(b->d_jac, B * f.nnz, double)
  if (has_cost) { TWB_ENSURE(b->d_cost, B, double) TWB_ENSURE(b->d_grad, B * f.n, double) }
#undef TWB_ENSURE
  // Pipelined in chunks of whole instance tiles: the H2D copy of chunk c+1 (copy-in stream), the kernels of chunk c
  // (b->stream + the two auxiliary streams) and the D2H copies of chunk c-1 (copy-out stream) overlap, so the call costs
  // what the larger of the two PCIe directions costs (the D2H of g + jac: 524 MB on config 2) plus one chunk of latency.
  const size_t group = 32 * (size_t)std::max(b->plan.nc_jac, 1);   // chunks hold whole groups of interleaved tiles
  const size_t chunk = ((size_t)std::max(32, b->e2e_chunk) + group - 1) / group * group;
  const size_t n_chunks = (B + chunk - 1) / chunk;
  if (!b->s_in && ((e = cudaStreamCreateWithFlags(&b->s_in, cudaStreamNonBlocking)) != cudaSuccess ||
                   (e = cudaStreamCreateWithFlags(&b->s_out, cudaStreamNonBlocking)) != cudaSuccess)) return CudaFail(e, "cudaStreamCreate");
  while (b->ev_chunk.size() < 2 * n_chunks) {
    cudaEvent_t ev; if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return CudaFail(e, "cudaEventCreate");
    b->ev_chunk.push_back(ev);
  }
  cudaStream_t s = b->stream;
  unsigned kflags = flags & (TWB_EVAL_G | TWB_EVAL_JAC);
  if (has_cost) kflags |= TWB_EVAL_COST;
  int launches = 0;
  twb::SetL2Window(b->use_l2_window ? &b->l2_window : nullptr);
  for (size_t c = 0; c < n_chunks; ++c) {
    const size_t off = c * chunk, nb = std::min(chunk, B - off), tile0 = off / 32;
    if ((e = cudaMemcpyAsync(b->d_x + off * f.n, x + off * f.n, sizeof(double) * nb * f.n, cudaMemcpyHostToDevice, b->s_in)) != cudaSuccess)
      return CudaFail(e, "H2D copy");
    cudaEventRecord(b->ev_chunk[2 * c], b->s_in);
    cudaStreamWaitEvent(s, b->ev_chunk[2 * c], 0);
    int rc = twb::LaunchEval(b->plan, b->d_x + off * f.n, b->d_XT + tile0 * (size_t)(f.n + 1) * 32, b->d_GT + tile0 * (size_t)std::max(f.m, 1) * 32,
                             b->d_FS ? b->d_FS + tile0 * (size_t)b->plan.n_dyn * 6 * b->plan.n_ee * 32 : nullptr, b->d_TD + tile0,
                             (flags & TWB_EVAL_G) ? b->d_g + off * f.m : nullptr, (flags & TWB_EVAL_JAC) ? b->d_jac + off * f.nnz : nullptr,
                             has_cost ? b->d_cost + off : nullptr, has_cost ? b->d_grad + off * f.n : nullptr, b->d_status + off,
                             b->d_terrain ? b->d_terrain + off : nullptr, f.spec.terrain, (int)nb, kflags, s, b->aux0, b->aux1, b->ev.data(), &launches);
    if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "kernel launch");
    cudaEventRecord(b->ev_chunk[2 * c + 1], s);
    cudaStreamWaitEvent(b->s_out, b->ev_chunk[2 * c + 1], 0);
    cudaStream_t o = b->s_out;
    if ((flags & TWB_EVAL_G) && g) cudaMemcpyAsync(g + off * f.m, b->d_g + off * f.m, sizeof(double) * nb * f.m, cudaMemcpyDeviceToHost, o);
    if ((flags & TWB_EVAL_JAC) && jac) cudaMemcpyAsync(jac + off * f.nnz, b->d_jac + off * f.nnz, sizeof(double) * nb * f.nnz, cudaMemcpyDeviceToHost, o);
    if (has_cost && cost) cudaMemcpyAsync(cost + off, b->d_cost + off, sizeof(double) * nb, cudaMemcpyDeviceToHost, o);
    if (has_cost && grad) cudaMemcpyAsync(grad + off * f.n, b->d_grad + off * f.n, sizeof(double) * nb * f.n, cudaMemcpyDeviceToHost, o);
    if (status) cudaMemcpyAsync(status + off, b->d_status + off, sizeof(int) * nb, cudaMemcpyDeviceToHost, o);
  }
  b->launches_last = launches;
  if ((e = cudaStreamSynchronize(b->s_out)) != cudaSuccess) return CudaFail(e, "evaluation");
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return CudaFail(e, "evaluation");
  if (!has_cost && (flags & TWB_EVAL_COST)) {  // Problem::EvaluateCostFunction without cost terms: 0
    if (cost) for (size_t i = 0; i < B; ++i) cost[i] = 0.0;
    if (grad) std::memset(grad, 0, sizeof(double) * B * f.n);
  }
  return TWB_OK;
}

}  // extern "C"
