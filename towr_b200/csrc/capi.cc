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

static_assert(TWB_STATE_DOUBLES == twb::kStateDoubles && twb::kStInitEE + 3 * TWB_MAX_EE == TWB_STATE_DOUBLES, "state record layout");

struct twb_problem {
  twb::Formulation f;
};

struct twb_batch {
  const twb_problem* prob = nullptr;
  int B = 0, device = 0;
  size_t ld = 0;                  // instances padded to a multiple of 32 (whole tiles of XT)
  twb::Plan plan{};
  std::vector<void*> owned;       // device allocations of the tables
  int* d_terrain = nullptr;       // per-instance terrain words (device_tables.h: TerrainWord; optional)
  std::vector<int> h_terrain;     // host copies of the terrain ids (empty: twb_spec.terrain) and of the grid_map indices
  std::vector<int> h_map_of;      // (empty: map 0) that d_terrain is packed from
  double* d_grid = nullptr;       // height grid of TWB_GRID_CSV (optional)
  float* d_gmap_pool = nullptr;   // elevation layers of TWB_GRID_MAP, back to back (optional)
  twb::GridMapDesc* d_gmaps = nullptr;   // one descriptor per layer
  double* d_XT = nullptr;         // [ld/32][n+1][32] instance-tiled iterates; row n == 0
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
  // twb_batch_lm_solve_device: the work arrays of the loop (one allocation, made by the first solve call) and the instantiated
  // solve graphs, one per argument set, cached like the evaluation graphs (up to 16, least recently used replaced, dropped
  // with them).  lm_stage: the host twin's device copies of its arguments (first host call).
  struct LmWork { double *g, *jac, *x_trial, *g_trial, *row_scale, *merit, *predicted, *nu; int* loop; };
  void* lm_work_mem = nullptr;
  LmWork lm_work{};
  double* lm_radius = nullptr;   // [2][B]: the trust radius and the last trial's max |d| (first trust-region solve)
  struct LmStage { double *x, *xl, *xu, *gl, *gu, *violation, *mu; int *status, *iterations, *counts, *loop_count; };
  void* lm_stage_mem = nullptr;
  LmStage lm_stage{};
  struct SolveGraph { const void* ptr[11]; twb_lm_solve_options opt; cudaGraphExec_t exec; unsigned long long used; };
  std::vector<SolveGraph> solve_graphs;
  int solve_instantiations = 0;   // graphs instantiated so far (twb_batch_lm_solve_graph_stats)
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
  for (auto& gr : b->solve_graphs) cudaGraphExecDestroy(gr.exec);
  b->solve_graphs.clear();
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
int NearestPlanesCore(twb_batch* b, const double* plan, const int* n_states, const int* poly_ranges, const int* poly_offsets, int n_polys,
                      const double* vertices, int* contact_set, cudaStream_t s) {
  int max_states = 0;
  twb_problem_footstep_plan_dims(b->prob, &max_states, nullptr);
  const int rc = twb::LaunchNearestPlanes(plan, n_states, max_states, b->prob->f.spec.n_ee, poly_offsets, n_polys, poly_ranges, vertices,
                                          contact_set, b->B, s);
  return rc != 0 ? CudaFail(static_cast<cudaError_t>(rc), "nearest-plane kernel launch") : TWB_OK;
}
// host arrays in, host contact sets out; poly_ranges may be null (every instance looks at all polygons)
int NearestPlanesHost(twb_batch* b, const double* plan, const int* n_states, const int* poly_ranges, const int* poly_offsets, int n_polys,
                      const double* vertices, int* contact_set) {
  if (!b || !plan || !n_states || !poly_offsets || !contact_set || n_polys < 0 || (n_polys > 0 && !vertices)) return Fail(TWB_ERR_INVALID, "null argument");
  for (int k = 0; k < n_polys; ++k) if (poly_offsets[k + 1] < poly_offsets[k] || poly_offsets[k] < 0) return Fail(TWB_ERR_INVALID, "polygon offsets must ascend");
  if (poly_ranges)
    for (int i = 0; i < b->B; ++i)
      if (poly_ranges[2 * i] < 0 || poly_ranges[2 * i + 1] < 0 || (long long)poly_ranges[2 * i] + poly_ranges[2 * i + 1] > n_polys)
        return Fail(TWB_ERR_INVALID, "polygon range outside the polygon list");
  int max_states = 0, V = 0;
  twb_problem_footstep_plan_dims(b->prob, &max_states, &V);
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const size_t B = b->B, n_ee = b->prob->f.spec.n_ee, n_vert = n_polys > 0 ? (size_t)poly_offsets[n_polys] : 0;
  double* d_plan = nullptr; int* d_count = nullptr; int* d_off = nullptr; double* d_vert = nullptr; int* d_out = nullptr; int* d_ranges = nullptr;
  // scratch buffers stay with the batch (twb_batch::scratch) and are reused by the next call
  if ((e = ScratchAlloc(b, 0, reinterpret_cast<void**>(&d_plan), sizeof(double) * B * max_states * V)) != cudaSuccess ||
      (e = ScratchAlloc(b, 1, reinterpret_cast<void**>(&d_count), sizeof(int) * B)) != cudaSuccess ||
      (e = ScratchAlloc(b, 2, reinterpret_cast<void**>(&d_off), sizeof(int) * (n_polys + 1))) != cudaSuccess ||
      (e = ScratchAlloc(b, 3, reinterpret_cast<void**>(&d_vert), sizeof(double) * 2 * std::max<size_t>(n_vert, 1))) != cudaSuccess ||
      (e = ScratchAlloc(b, 4, reinterpret_cast<void**>(&d_out), sizeof(int) * B * max_states * n_ee)) != cudaSuccess ||
      (poly_ranges && (e = ScratchAlloc(b, 5, reinterpret_cast<void**>(&d_ranges), sizeof(int) * 2 * B)) != cudaSuccess)) return CudaFail(e, "cudaMalloc");
  cudaStream_t s = b->stream;
  cudaMemcpyAsync(d_plan, plan, sizeof(double) * B * max_states * V, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(d_count, n_states, sizeof(int) * B, cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(d_off, poly_offsets, sizeof(int) * (n_polys + 1), cudaMemcpyHostToDevice, s);
  if (n_vert) cudaMemcpyAsync(d_vert, vertices, sizeof(double) * 2 * n_vert, cudaMemcpyHostToDevice, s);
  if (poly_ranges) cudaMemcpyAsync(d_ranges, poly_ranges, sizeof(int) * 2 * B, cudaMemcpyHostToDevice, s);
  int rc = NearestPlanesCore(b, d_plan, d_count, d_ranges, d_off, n_polys, d_vert, d_out, s);
  if (rc == TWB_OK) cudaMemcpyAsync(contact_set, d_out, sizeof(int) * B * max_states * n_ee, cudaMemcpyDeviceToHost, s);
  e = cudaStreamSynchronize(s);
  if (rc != TWB_OK) return rc;
  if (e != cudaSuccess) return CudaFail(e, "nearest-plane lookup");
  return TWB_OK;
}
int NearestPlanesDevice(twb_batch* b, const double* plan, const int* n_states, const int* poly_ranges, const int* poly_offsets, int n_polys,
                        const double* vertices, int* contact_set, void* stream) {
  if (!b || !plan || !n_states || !poly_offsets || !contact_set || n_polys < 0 || (n_polys > 0 && !vertices)) return Fail(TWB_ERR_INVALID, "null argument");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  return NearestPlanesCore(b, plan, n_states, poly_ranges, poly_offsets, n_polys, vertices, contact_set, static_cast<cudaStream_t>(stream));
}

// d_terrain from the host copies of the terrain ids and grid_map indices (device_tables.h: TerrainWord); none of either:
// no per-instance words, every instance evaluates twb_spec.terrain
int UploadTerrainWords(twb_batch* b) {
  if (b->h_terrain.empty() && b->h_map_of.empty()) { cudaFree(b->d_terrain); b->d_terrain = nullptr; return TWB_OK; }
  std::vector<int> words(b->B);
  for (int i = 0; i < b->B; ++i)
    words[i] = twb::TerrainWord(b->h_terrain.empty() ? b->prob->f.spec.terrain : b->h_terrain[i], b->h_map_of.empty() ? 0 : b->h_map_of[i]);
  cudaError_t e;
  if (!b->d_terrain && (e = cudaMalloc(&b->d_terrain, sizeof(int) * b->B)) != cudaSuccess) return CudaFail(e, "cudaMalloc");
  if ((e = cudaMemcpy(b->d_terrain, words.data(), sizeof(int) * b->B, cudaMemcpyHostToDevice)) != cudaSuccess) return CudaFail(e, "cudaMemcpy");
  return TWB_OK;
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
int twb_problem_state_instances(const twb_problem* p, int n_states, const double* states, double* x0, double* xl, double* xu, double* gl,
                                double* gu) {
  if (!p || !states || n_states <= 0) return Fail(TWB_ERR_INVALID, "bad argument");
  const size_t n = (size_t)p->f.n, m = (size_t)p->f.m;
  for (int i = 0; i < n_states; ++i) {
    int rc = p->f.StateInstance(states + (size_t)TWB_STATE_DOUBLES * i, x0 ? x0 + i * n : nullptr, xl ? xl + i * n : nullptr,
                                xu ? xu + i * n : nullptr, gl ? gl + i * m : nullptr, gu ? gu + i * m : nullptr);
    if (rc != TWB_OK) return Fail(rc, "state instance");
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
  TWB_UP(state_vars) TWB_UP(base_z_rows)
#undef TWB_UP
  if ((e = Upload(p->f.g_lower, &b->plan.g_lower, &b->owned)) != cudaSuccess || (e = Upload(p->f.g_upper, &b->plan.g_upper, &b->owned)) != cudaSuccess) {
    twb_batch_destroy(b);
    return CudaFail(e, "table upload");
  }
  if (std::getenv("TWB_PROFILE") && !g_prof_on) { g_prof_on = true; twb::g_after_launch = ProfHook; std::atexit(ProfReport); }
  if (g_prof_on) std::fprintf(stderr, "[twb profile] n=%d m=%d nnz=%d\n", b->plan.n, b->plan.m, b->plan.nnz);
  if (const char* v = std::getenv("TWB_E2E_CHUNK")) b->e2e_chunk = std::max(32, std::atoi(v));
  if (const char* v = std::getenv("TWB_GRAPH")) b->use_graphs = std::atoi(v) != 0;
  if (const char* v = std::getenv("TWB_EVAL_CHUNK")) b->eval_chunk = (size_t)std::max(0, std::atoi(v));
  // whole groups of nc interleaved tiles (kernels.cu: TileInstance); nc = 1 unless the Jacobian row length is not a multiple of 4
  const size_t group = 32 * (size_t)std::max(b->plan.nc_jac, 1);
  b->ld = ((size_t)batch_size + group - 1) / group * group;
  const size_t xt_bytes = (size_t)(b->plan.n + 1) * b->ld * sizeof(double);
  if ((e = cudaMalloc(reinterpret_cast<void**>(&b->d_XT), xt_bytes)) != cudaSuccess ||
      (e = cudaMemset(b->d_XT, 0, xt_bytes)) != cudaSuccess) {
    twb_batch_destroy(b);
    return CudaFail(e, "state allocation");
  }
  if (b->plan.n_phase_defs > 0 && b->plan.n_dyn > 0 &&
      (e = cudaMalloc(reinterpret_cast<void**>(&b->d_FS), (size_t)b->plan.n_dyn * 6 * b->plan.n_ee * b->ld * sizeof(double))) != cudaSuccess) {
    twb_batch_destroy(b);
    return CudaFail(e, "state allocation");
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
  for (void* p : b->owned) cudaFree(p);
  for (auto& sc : b->scratch) cudaFree(sc.first);
  for (auto& t : b->post_tables) cudaFree(t.mem);
  cudaFree(b->lm_work_mem); cudaFree(b->lm_stage_mem); cudaFree(b->lm_radius);
  cudaFree(b->d_terrain); cudaFree(b->d_grid); cudaFree(b->d_gmap_pool); cudaFree(b->d_gmaps); cudaFree(b->d_XT); cudaFree(b->d_FS);
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
  if (!terrain_ids) { b->h_terrain.clear(); return UploadTerrainWords(b); }
  for (int i = 0; i < b->B; ++i)
    if (terrain_ids[i] < 0 || terrain_ids[i] > TWB_GRID_MAP) return Fail(TWB_ERR_INVALID, "unknown terrain id");
  b->h_terrain.assign(terrain_ids, terrain_ids + b->B);
  return UploadTerrainWords(b);
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
  const int sizes[2] = {size_x, size_y};
  const double geometry[3] = {resolution, pos_x, pos_y};
  return twb_batch_set_grid_maps(b, heights ? 1 : 0, heights, sizes, geometry, nullptr);
}

int twb_batch_set_grid_maps(twb_batch* b, int n_maps, const float* heights, const int* sizes, const double* geometry, const int* map_of_instance) {
  if (!b) return Fail(TWB_ERR_INVALID, "null batch");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  float* pool = nullptr; twb::GridMapDesc* table = nullptr;
  std::vector<int> map_of;
  if (n_maps < 0 || n_maps > twb::kMaxGridMaps) return Fail(TWB_ERR_INVALID, "bad number of grid maps");
  if (heights && n_maps > 0) {   // checked and uploaded before the previous maps are released: a failed call keeps them
    if (!sizes || !geometry) return Fail(TWB_ERR_INVALID, "null argument");
    std::vector<twb::GridMapDesc> desc(n_maps);
    long long cells = 0;
    for (int k = 0; k < n_maps; ++k) {
      const int sx = sizes[2 * k], sy = sizes[2 * k + 1];
      const double res = geometry[3 * k], px = geometry[3 * k + 1], py = geometry[3 * k + 2];
      if (sx <= 0 || sy <= 0 || (long long)sx * sy > (1ll << 28) || !(res > 0.0) || !std::isfinite(res) || !std::isfinite(px) || !std::isfinite(py))
        return Fail(TWB_ERR_INVALID, "bad grid map geometry");
      desc[k] = twb::GridMapDesc{cells, sx, sy, res, px, py};
      cells += (long long)sx * sy;
    }
    if (map_of_instance) {
      for (int i = 0; i < b->B; ++i)
        if (map_of_instance[i] < 0 || map_of_instance[i] >= n_maps) return Fail(TWB_ERR_INVALID, "grid map index out of range");
      map_of.assign(map_of_instance, map_of_instance + b->B);
    }
    if ((e = cudaMalloc(reinterpret_cast<void**>(&pool), sizeof(float) * (size_t)cells)) != cudaSuccess ||
        (e = cudaMalloc(reinterpret_cast<void**>(&table), sizeof(twb::GridMapDesc) * n_maps)) != cudaSuccess ||
        (e = cudaMemcpy(pool, heights, sizeof(float) * (size_t)cells, cudaMemcpyHostToDevice)) != cudaSuccess ||
        (e = cudaMemcpy(table, desc.data(), sizeof(twb::GridMapDesc) * n_maps, cudaMemcpyHostToDevice)) != cudaSuccess) {
      cudaFree(pool); cudaFree(table);
      return CudaFail(e, "grid map upload");
    }
  } else {
    n_maps = 0;
  }
  DropGraphs(b);
  cudaFree(b->d_gmap_pool); cudaFree(b->d_gmaps);
  b->d_gmap_pool = pool; b->d_gmaps = table;
  b->plan.gmap_pool = pool; b->plan.gmaps = table; b->plan.n_gmaps = n_maps;
  b->h_map_of.swap(map_of);
  return UploadTerrainWords(b);
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

int twb_batch_state_instances_device(twb_batch* b, const double* states, double* x0, double* x_lower, double* x_upper, double* g_lower,
                                     double* g_upper, void* stream) {
  if (!b || !states) return Fail(TWB_ERR_INVALID, "null argument");
  if (!x0 && !x_lower && !x_upper && !g_lower && !g_upper) return Fail(TWB_ERR_INVALID, "no output requested");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb::Formulation& f = b->prob->f;
  int rc = twb::LaunchStateInstances(b->plan, f.tables.goal_setup, states, b->d_terrain, f.spec.terrain, x0, x_lower, x_upper, g_lower, g_upper, b->B,
                                     static_cast<cudaStream_t>(stream));
  if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "state-instance kernel launch");
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
  return NearestPlanesHost(b, plan, n_states, nullptr, poly_offsets, n_polys, vertices, contact_set);
}

int twb_batch_nearest_planes_device(twb_batch* b, const double* plan, const int* n_states, const int* poly_offsets, int n_polys,
                                    const double* vertices, int* contact_set, void* stream) {
  return NearestPlanesDevice(b, plan, n_states, nullptr, poly_offsets, n_polys, vertices, contact_set, stream);
}

int twb_batch_nearest_planes_ranges_host(twb_batch* b, const double* plan, const int* n_states, const int* poly_ranges,
                                         const int* poly_offsets, int n_polys, const double* vertices, int* contact_set) {
  if (!poly_ranges) return Fail(TWB_ERR_INVALID, "null argument");
  return NearestPlanesHost(b, plan, n_states, poly_ranges, poly_offsets, n_polys, vertices, contact_set);
}

int twb_batch_nearest_planes_ranges_device(twb_batch* b, const double* plan, const int* n_states, const int* poly_ranges,
                                           const int* poly_offsets, int n_polys, const double* vertices, int* contact_set,
                                           void* stream) {
  if (!poly_ranges) return Fail(TWB_ERR_INVALID, "null argument");
  return NearestPlanesDevice(b, plan, n_states, poly_ranges, poly_offsets, n_polys, vertices, contact_set, stream);
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
  if (flags & (TWB_EVAL_G | TWB_EVAL_JAC)) n += twb::OutKernelsPerEval(p, flags);   // DynOut [+ DynTailOut] + RomNodeOut
  if ((flags & (TWB_EVAL_G | TWB_EVAL_JAC)) && p.n_phase_units > 0) n += 1;   // PhaseJac
  if (want_cost) n += 1;
  {   // large batches are evaluated chunk after chunk (twb_batch::eval_chunk)
    const size_t B = (size_t)b->B, chunk = EvalChunk(b);
    n *= (int)((B + chunk - 1) / chunk);
  }
  return n;
}

}  // extern "C"

// The kernels of one evaluation (what twb_batch_eval_device enqueues without its graph cache): the whole batch, or chunk after
// chunk (twb_batch::eval_chunk), on s0 and the batch's two auxiliary streams
static int EnqueueEval(twb_batch* b, const double* x, double* g, double* jac, double* cost, double* grad, int* status, unsigned kflags,
                       cudaStream_t s0, int* launches) {
  const twb::Formulation& f = b->prob->f;
  const size_t B = (size_t)b->B;
  const size_t chunk = EvalChunk(b);
  const size_t n = f.n, m = f.m;
  for (size_t off = 0; off < B; off += chunk) {
    const size_t nb = std::min(chunk, B - off), t0 = off / 32;
    const int rc = twb::LaunchEval(b->plan, x + off * n, b->d_XT + t0 * (n + 1) * 32,
                                   b->d_FS ? b->d_FS + t0 * (size_t)b->plan.n_dyn * 6 * b->plan.n_ee * 32 : nullptr,
                                   g ? g + off * m : nullptr, jac ? jac + off * (size_t)f.nnz : nullptr, cost ? cost + off : nullptr,
                                   grad ? grad + off * n : nullptr, status ? status + off : nullptr,
                                   b->d_terrain ? b->d_terrain + off : nullptr, f.spec.terrain, (int)nb, kflags, s0, b->aux0, b->aux1, b->ev.data(),
                                   launches);
    if (rc != 0) return rc;
  }
  return 0;
}

extern "C" {

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
  auto enqueue = [&](cudaStream_t s0) -> int {
    return EnqueueEval(b, x, g, jac, cost, grad, status, kflags, s0, &launches);
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

// The first call of the step family on a batch uploads what the solver kernels read besides their arguments: the pattern, its
// transpose (entries of column j in ascending row order: what a stable sort by column yields), the row / column orders, the
// 16-bit index arrays when they fit, and the problem's variable and constraint bounds.  Later calls find it in place.
static int LmPatternReady(twb_batch* b) {
  cudaError_t e;
  const twb::Formulation& f = b->prob->f;
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
  return TWB_OK;
}

// twb_batch_lm_step_device, twb_batch_lm_step_bounds_device and twb_batch_lm_trial_device (trial non-null: mu unused):
// g_lower / g_upper null = the problem's constraint bounds
static int LmStepDevice(twb_batch* b, double* x, const double* g, const double* jac, const double* x_lower, const double* x_upper,
                        const double* g_lower, const double* g_upper, double mu, double cap, int cg_iters, double* violation,
                        const twb::LmTrialArgs* trial, void* stream) {
  if (!b || !x || !g || !jac) return Fail(TWB_ERR_INVALID, "null argument");
  if ((x_lower == nullptr) != (x_upper == nullptr)) return Fail(TWB_ERR_INVALID, "x_lower and x_upper: both or neither");
  if ((g_lower == nullptr) != (g_upper == nullptr)) return Fail(TWB_ERR_INVALID, "g_lower and g_upper: both or neither");
  if (!(mu >= 0.0) || !(cap > 0.0) || cg_iters < 0 || cg_iters > 10000) return Fail(TWB_ERR_INVALID, "bad solver parameter");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb::Formulation& f = b->prob->f;
  if (twb::LmSharedBytes(f.n, f.m) > 200 * 1024) return Fail(TWB_ERR_UNSUPPORTED, "problem too large for the shared-memory solver step");
  int rc = LmPatternReady(b);
  if (rc != TWB_OK) return rc;
  const bool own = x_lower != nullptr, own_g = g_lower != nullptr;
  rc = twb::LaunchLmStep(b->lm_pat, f.n, f.m, f.nnz, x, g, jac, own ? x_lower : b->d_xl, own ? x_upper : b->d_xu, own ? (size_t)f.n : 0,
                         own_g ? g_lower : b->lm_pat.g_lower, own_g ? g_upper : b->lm_pat.g_upper, own_g ? (size_t)f.m : 0, mu, cap,
                         cg_iters, violation, trial, b->B, static_cast<cudaStream_t>(stream));
  if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "solver step launch");
  return TWB_OK;
}

int twb_batch_lm_step_device(twb_batch* b, double* x, const double* g, const double* jac, const double* x_lower, const double* x_upper,
                             double mu, double cap, int cg_iters, double* violation, void* stream) {
  return LmStepDevice(b, x, g, jac, x_lower, x_upper, nullptr, nullptr, mu, cap, cg_iters, violation, nullptr, stream);
}

int twb_batch_lm_step_bounds_device(twb_batch* b, double* x, const double* g, const double* jac, const double* x_lower, const double* x_upper,
                                    const double* g_lower, const double* g_upper, double mu, double cap, int cg_iters, double* violation,
                                    void* stream) {
  return LmStepDevice(b, x, g, jac, x_lower, x_upper, g_lower, g_upper, mu, cap, cg_iters, violation, nullptr, stream);
}

static_assert(TWB_LM_RUNNING == twb::kLmRunning && TWB_LM_CONVERGED == twb::kLmConverged && TWB_LM_STALLED == twb::kLmStalled &&
              TWB_LM_NONFINITE == twb::kLmNonFinite, "solve status codes");

int twb_batch_lm_trial_device(twb_batch* b, const double* x, const double* g, const double* jac, const double* x_lower, const double* x_upper,
                              const double* g_lower, const double* g_upper, const double* mu, double cap, int cg_iters, double tol,
                              int* solve_status, double* x_trial, double* row_scale, double* merit, double* predicted, double* violation,
                              void* stream) {
  if (!mu || !solve_status || !x_trial || !row_scale || !merit || !predicted) return Fail(TWB_ERR_INVALID, "null argument");
  if (!(tol >= 0.0)) return Fail(TWB_ERR_INVALID, "bad tolerance");
  const twb::LmTrialArgs trial{mu, tol, solve_status, x_trial, row_scale, merit, predicted};
  // x is only read by the trial kernel
  return LmStepDevice(b, const_cast<double*>(x), g, jac, x_lower, x_upper, g_lower, g_upper, 0.0, cap, cg_iters, violation, &trial, stream);
}

int twb_batch_lm_accept_device(twb_batch* b, double* x, const double* x_trial, const double* g_trial, const double* g_lower,
                               const double* g_upper, const double* row_scale, const double* merit, const double* predicted, double* mu,
                               double* nu, int* solve_status, int* iterations, double eta, double mu_min, double mu_max, void* stream) {
  if (!b || !x || !x_trial || !g_trial || !row_scale || !merit || !predicted || !mu || !nu || !solve_status || !iterations)
    return Fail(TWB_ERR_INVALID, "null argument");
  if ((g_lower == nullptr) != (g_upper == nullptr)) return Fail(TWB_ERR_INVALID, "g_lower and g_upper: both or neither");
  if (!(eta >= 0.0 && eta < 1.0) || !(mu_min > 0.0 && mu_min <= mu_max)) return Fail(TWB_ERR_INVALID, "bad solver parameter");
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb::Formulation& f = b->prob->f;
  int rc = LmPatternReady(b);
  if (rc != TWB_OK) return rc;
  const bool own_g = g_lower != nullptr;
  rc = twb::LaunchLmAccept(f.n, f.m, x, x_trial, g_trial, own_g ? g_lower : b->lm_pat.g_lower, own_g ? g_upper : b->lm_pat.g_upper,
                           own_g ? (size_t)f.m : 0, row_scale, merit, predicted, mu, nu, solve_status, iterations, eta, mu_min, mu_max,
                           nullptr, nullptr, 0.0, b->B, static_cast<cudaStream_t>(stream));
  if (rc != 0) return CudaFail(static_cast<cudaError_t>(rc), "solver accept launch");
  return TWB_OK;
}

void twb_lm_solve_options_default(twb_lm_solve_options* o) {
  if (o) *o = twb_lm_solve_options{1e-2, 0.1, 1e-6, 1e-4, 1e-12, 1e10, 25, 60, TWB_LM_STEP_CAP, 1e3};
}

// the options as a graph-cache key, field by field (the struct has padding after step_rule)
static bool SameOptions(const twb_lm_solve_options& a, const twb_lm_solve_options& b) {
  return a.mu0 == b.mu0 && a.cap == b.cap && a.tol == b.tol && a.eta == b.eta && a.mu_min == b.mu_min && a.mu_max == b.mu_max &&
         a.cg_iters == b.cg_iters && a.max_iters == b.max_iters && a.step_rule == b.step_rule && a.radius_max == b.radius_max;
}

// ---- twb_batch_lm_solve_device: the solve loop as one CUDA graph with a WHILE node --------------------------------------
// the arguments of one solve; together they are the key of the graph cache
struct LmSolveCall {
  double* x; const double *xl, *xu, *gl, *gu;
  int *status, *iterations; double *violation, *mu; int *counts, *loop_count;
  twb_lm_solve_options opt;
  void Key(const void* (&k)[11]) const {
    const void* v[11] = {x, xl, xu, gl, gu, status, iterations, violation, mu, counts, loop_count};
    std::copy(v, v + 11, k);
  }
};

// the checks of the device call and its host twin that need no device
static int LmSolveArgs(const twb_batch* b, const LmSolveCall& c) {
  if (!b || !c.x || !c.status || !c.iterations || !c.violation || !c.mu) return Fail(TWB_ERR_INVALID, "null argument");
  if ((c.xl == nullptr) != (c.xu == nullptr)) return Fail(TWB_ERR_INVALID, "x_lower and x_upper: both or neither");
  if ((c.gl == nullptr) != (c.gu == nullptr)) return Fail(TWB_ERR_INVALID, "g_lower and g_upper: both or neither");
  const twb_lm_solve_options& o = c.opt;
  if (o.max_iters < 0) return Fail(TWB_ERR_INVALID, "max_iters < 0");
  if (!(o.tol >= 0.0)) return Fail(TWB_ERR_INVALID, "bad tolerance");
  if (!(o.eta >= 0.0 && o.eta < 1.0) || !(o.mu_min > 0.0 && o.mu_min <= o.mu_max) || !(o.mu0 > 0.0) || !(o.cap > 0.0) || o.cg_iters < 0 ||
      o.cg_iters > 10000)
    return Fail(TWB_ERR_INVALID, "bad solver parameter");
  if (o.step_rule != TWB_LM_STEP_CAP && o.step_rule != TWB_LM_STEP_TRUST) return Fail(TWB_ERR_INVALID, "unknown step_rule");
  if (o.step_rule == TWB_LM_STEP_TRUST && !(o.radius_max >= o.cap)) return Fail(TWB_ERR_INVALID, "radius_max < cap or NaN");
  if (g_prof_on) return Fail(TWB_ERR_UNSUPPORTED, "TWB_PROFILE records events around every kernel, which a device-side loop cannot hold");
  const twb::Formulation& f = b->prob->f;
  if (twb::LmSharedBytes(f.n, f.m) > 200 * 1024) return Fail(TWB_ERR_UNSUPPORTED, "problem too large for the shared-memory solver step");
  return TWB_OK;
}

// the loop's work arrays, one allocation (every array at a 256-byte boundary), made on the first solve call
static int LmWorkReady(twb_batch* b) {
  if (b->lm_work_mem) return TWB_OK;
  const twb::Formulation& f = b->prob->f;
  const size_t B = b->B;
  auto up = [](size_t bytes) { return (bytes + 255) & ~(size_t)255; };
  const size_t counts[8] = {B * f.m, B * f.nnz, B * f.n, B * f.m, B * f.m, B, B, B};   // g, jac, x_trial, g_trial, row_scale, merit, predicted, nu
  size_t off[9] = {0};
  for (int k = 0; k < 8; ++k) off[k + 1] = off[k] + up(sizeof(double) * counts[k]);
  void* mem = nullptr;
  cudaError_t e = cudaMalloc(&mem, off[8] + up(sizeof(int) * twb::kLoopInts));
  if (e != cudaSuccess) return CudaFail(e, "cudaMalloc");
  char* p = static_cast<char*>(mem);
  double* a[8];
  for (int k = 0; k < 8; ++k) a[k] = reinterpret_cast<double*>(p + off[k]);
  b->lm_work = {a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], reinterpret_cast<int*>(p + off[8])};
  b->lm_work_mem = mem;
  return TWB_OK;
}

// the trust-region rule's radius and step_norm [B] each, made on the first trust-region solve
static int LmRadiusReady(twb_batch* b) {
  if (b->lm_radius) return TWB_OK;
  cudaError_t e = cudaMalloc(&b->lm_radius, sizeof(double) * 2 * (size_t)b->B);
  if (e != cudaSuccess) { b->lm_radius = nullptr; return CudaFail(e, "cudaMalloc"); }
  return TWB_OK;
}

// Captures the solve graph of `c`:
//   init -> WHILE { eval(G|JAC at x) -> trial -> eval(G at x_trial) -> accept -> count + condition } -> eval(G|JAC at x) ->
//   trial with cg_iters = 0 -> count into the caller's outputs
// The start and the tail are captured into the graph around the WHILE node, the body into the node's body graph.  The
// evaluations are captured as kernels, as twb_batch_eval_device enqueues them without its graph cache (three streams joined by
// events, RomNodeOut with programmatic dependent launch: both instantiate inside the conditional body on the B200).
static cudaError_t CaptureSolveGraph(twb_batch* b, const LmSolveCall& c, cudaGraph_t* out) {
  const twb::Formulation& f = b->prob->f;
  const twb_batch::LmWork& w = b->lm_work;
  const int B = b->B;
  const twb_lm_solve_options& o = c.opt;
  cudaStream_t s = b->stream;
  const bool own = c.xl != nullptr, own_g = c.gl != nullptr;
  const double *xl = own ? c.xl : b->d_xl, *xu = own ? c.xu : b->d_xu;
  const double *gl = own_g ? c.gl : b->lm_pat.g_lower, *gu = own_g ? c.gu : b->lm_pat.g_upper;
  const size_t xs = own ? (size_t)f.n : 0, gs = own_g ? (size_t)f.m : 0;
  const bool trust = o.step_rule == TWB_LM_STEP_TRUST;
  double* radius = trust ? b->lm_radius : nullptr;
  double* step_norm = trust ? b->lm_radius + B : nullptr;
  const twb::LmTrialArgs trial{c.mu, o.tol, c.status, w.x_trial, w.row_scale, w.merit, w.predicted, radius, step_norm};
  // the tail only measures (cg_iters = 0: no step under either rule); the cap rule's trial there leaves step_norm as the
  // last loop trial wrote it
  const twb::LmTrialArgs tail{c.mu, o.tol, c.status, w.x_trial, w.row_scale, w.merit, w.predicted, nullptr, nullptr};
  auto eval = [&](const double* x, double* g, double* jac, unsigned flags) {
    return EnqueueEval(b, x, g, jac, nullptr, nullptr, nullptr, flags, s, nullptr);
  };
  auto trial_step = [&](int cg_iters, const twb::LmTrialArgs* args) {
    return twb::LaunchLmStep(b->lm_pat, f.n, f.m, f.nnz, c.x, w.g, w.jac, xl, xu, xs, gl, gu, gs, 0.0, o.cap, cg_iters, c.violation, args, B, s);
  };
  cudaGraph_t graph = nullptr;
  cudaGraphConditionalHandle cond = 0;
  cudaGraphNodeParams loop{};
  cudaError_t e = cudaGraphCreate(&graph, 0);
  if (e == cudaSuccess) e = cudaGraphConditionalHandleCreate(&cond, graph, 0, 0);
  if (e == cudaSuccess) e = cudaStreamBeginCaptureToGraph(s, graph, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed);
  if (e == cudaSuccess) {   // the start, the WHILE node after it, the tail after that
    int rc = twb::LaunchLmSolveInit(B, o.mu0, c.mu, w.nu, c.status, c.iterations, o.cap, radius, step_norm, w.loop, o.max_iters, cond, s);
    cudaStreamCaptureStatus cs;
    const cudaGraphNode_t* deps = nullptr;
    size_t n_deps = 0;
    cudaGraphNode_t node = nullptr;
    if (rc == 0) rc = cudaStreamGetCaptureInfo(s, &cs, nullptr, nullptr, &deps, &n_deps);
    if (rc == 0) {
      loop.type = cudaGraphNodeTypeConditional;
      loop.conditional.handle = cond;
      loop.conditional.type = cudaGraphCondTypeWhile;
      loop.conditional.size = 1;
      rc = cudaGraphAddNode(&node, graph, deps, n_deps, &loop);
    }
    if (rc == 0) rc = cudaStreamUpdateCaptureDependencies(s, &node, 1, cudaStreamSetCaptureDependencies);
    if (rc == 0) rc = eval(c.x, w.g, w.jac, TWB_EVAL_G | TWB_EVAL_JAC);
    if (rc == 0) rc = trial_step(0, &tail);
    if (rc == 0) rc = twb::LaunchLmCount(B, c.status, w.loop, o.max_iters, cond, false, c.counts, c.loop_count, s);
    cudaGraph_t captured = nullptr;
    e = cudaStreamEndCapture(s, &captured);
    if (rc != 0) e = static_cast<cudaError_t>(rc);
  }
  if (e == cudaSuccess) e = cudaStreamBeginCaptureToGraph(s, loop.conditional.phGraph_out[0], nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed);
  if (e == cudaSuccess) {   // the body
    int rc = eval(c.x, w.g, w.jac, TWB_EVAL_G | TWB_EVAL_JAC);
    if (rc == 0) rc = trial_step(o.cg_iters, &trial);
    if (rc == 0) rc = eval(w.x_trial, w.g_trial, nullptr, TWB_EVAL_G);
    if (rc == 0)
      rc = twb::LaunchLmAccept(f.n, f.m, c.x, w.x_trial, w.g_trial, gl, gu, gs, w.row_scale, w.merit, w.predicted, c.mu, w.nu, c.status,
                               c.iterations, o.eta, o.mu_min, o.mu_max, radius, step_norm, o.radius_max, B, s);
    if (rc == 0) rc = twb::LaunchLmCount(B, c.status, w.loop, o.max_iters, cond, true, nullptr, nullptr, s);
    cudaGraph_t captured = nullptr;
    e = cudaStreamEndCapture(s, &captured);
    if (rc != 0) e = static_cast<cudaError_t>(rc);
  }
  if (e != cudaSuccess) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    return e;
  }
  *out = graph;
  return cudaSuccess;
}

// the instantiated graph of `c`: from the cache, or captured and instantiated
static int SolveGraph(twb_batch* b, const LmSolveCall& c, cudaGraphExec_t* exec) {
  const void* key[11];
  c.Key(key);
  for (auto& gr : b->solve_graphs)
    if (std::equal(key, key + 11, gr.ptr) && SameOptions(gr.opt, c.opt)) {
      gr.used = ++b->graph_clock; *exec = gr.exec; return TWB_OK;
    }
  cudaGraph_t graph = nullptr;
  cudaError_t e = CaptureSolveGraph(b, c, &graph);
  if (e == cudaSuccess) {
    e = cudaGraphInstantiate(exec, graph, 0);
    cudaGraphDestroy(graph);
  }
  if (e != cudaSuccess) { cudaGetLastError(); return CudaFail(e, "solve graph"); }
  ++b->solve_instantiations;
  if (b->solve_graphs.size() >= 16) {   // replace the least recently used
    size_t lru = 0;
    for (size_t i = 1; i < b->solve_graphs.size(); ++i) if (b->solve_graphs[i].used < b->solve_graphs[lru].used) lru = i;
    cudaGraphExecDestroy(b->solve_graphs[lru].exec);
    b->solve_graphs.erase(b->solve_graphs.begin() + lru);
  }
  b->solve_graphs.push_back({{}, c.opt, *exec, ++b->graph_clock});
  std::copy(key, key + 11, b->solve_graphs.back().ptr);
  return TWB_OK;
}

static int LmSolveCore(twb_batch* b, const LmSolveCall& c, cudaStream_t stream) {
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if ((e = cudaStreamIsCapturing(stream, &cs)) != cudaSuccess) { cudaGetLastError(); return CudaFail(e, "cudaStreamIsCapturing"); }
  if (cs != cudaStreamCaptureStatusNone) return Fail(TWB_ERR_UNSUPPORTED, "the stream is being captured: a solve cannot be captured into a graph");
  int rc = LmPatternReady(b);
  if (rc == TWB_OK) rc = LmWorkReady(b);
  if (rc == TWB_OK && c.opt.step_rule == TWB_LM_STEP_TRUST) rc = LmRadiusReady(b);
  cudaGraphExec_t exec = nullptr;
  if (rc == TWB_OK) rc = SolveGraph(b, c, &exec);
  if (rc != TWB_OK) return rc;
  if ((e = cudaGraphLaunch(exec, stream)) != cudaSuccess) return CudaFail(e, "cudaGraphLaunch");
  return TWB_OK;
}

int twb_batch_lm_solve_device(twb_batch* b, double* x, const double* x_lower, const double* x_upper, const double* g_lower,
                              const double* g_upper, const twb_lm_solve_options* opt, int* solve_status, int* iterations,
                              double* violation, double* mu, int* status_counts, int* loop_count, void* stream) {
  if (!opt) return Fail(TWB_ERR_INVALID, "null argument");
  const LmSolveCall c{x, x_lower, x_upper, g_lower, g_upper, solve_status, iterations, violation, mu, status_counts, loop_count, *opt};
  const int rc = LmSolveArgs(b, c);
  return rc != TWB_OK ? rc : LmSolveCore(b, c, static_cast<cudaStream_t>(stream));
}

int twb_batch_lm_solve_host(twb_batch* b, double* x, const double* x_lower, const double* x_upper, const double* g_lower,
                            const double* g_upper, const twb_lm_solve_options* opt, int* solve_status, int* iterations,
                            double* violation, double* mu, int* status_counts, int* loop_count) {
  if (!opt) return Fail(TWB_ERR_INVALID, "null argument");
  const LmSolveCall h{x, x_lower, x_upper, g_lower, g_upper, solve_status, iterations, violation, mu, status_counts, loop_count, *opt};
  int rc = LmSolveArgs(b, h);
  if (rc != TWB_OK) return rc;
  cudaError_t e = cudaSetDevice(b->device);
  if (e != cudaSuccess) return CudaFail(e, "cudaSetDevice");
  const twb::Formulation& f = b->prob->f;
  const size_t B = b->B, xb = sizeof(double) * B * f.n, gb = sizeof(double) * B * f.m;
  if (!b->lm_stage_mem) {   // x, x bounds, g bounds, violation, mu, status, iterations, counts, loop count: one allocation
    auto up = [](size_t bytes) { return (bytes + 255) & ~(size_t)255; };
    const size_t sizes[11] = {xb, xb, xb, gb, gb, sizeof(double) * B, sizeof(double) * B, sizeof(int) * B, sizeof(int) * B, sizeof(int) * 4, sizeof(int)};
    size_t off[12] = {0};
    for (int k = 0; k < 11; ++k) off[k + 1] = off[k] + up(sizes[k]);
    void* mem = nullptr;
    if ((e = cudaMalloc(&mem, off[11])) != cudaSuccess) return CudaFail(e, "cudaMalloc");
    char* p = static_cast<char*>(mem);
    auto d = [&](int k) { return reinterpret_cast<double*>(p + off[k]); };
    auto i = [&](int k) { return reinterpret_cast<int*>(p + off[k]); };
    b->lm_stage = {d(0), d(1), d(2), d(3), d(4), d(5), d(6), i(7), i(8), i(9), i(10)};
    b->lm_stage_mem = mem;
  }
  const twb_batch::LmStage& st = b->lm_stage;
  cudaStream_t s = b->stream;
  cudaMemcpyAsync(st.x, x, xb, cudaMemcpyHostToDevice, s);
  if (x_lower) { cudaMemcpyAsync(st.xl, x_lower, xb, cudaMemcpyHostToDevice, s); cudaMemcpyAsync(st.xu, x_upper, xb, cudaMemcpyHostToDevice, s); }
  if (g_lower) { cudaMemcpyAsync(st.gl, g_lower, gb, cudaMemcpyHostToDevice, s); cudaMemcpyAsync(st.gu, g_upper, gb, cudaMemcpyHostToDevice, s); }
  const LmSolveCall c{st.x, x_lower ? st.xl : nullptr, x_lower ? st.xu : nullptr, g_lower ? st.gl : nullptr, g_lower ? st.gu : nullptr, st.status,
                      st.iterations, st.violation, st.mu, status_counts ? st.counts : nullptr, loop_count ? st.loop_count : nullptr, *opt};
  rc = LmSolveCore(b, c, s);
  if (rc == TWB_OK) {
    cudaMemcpyAsync(x, st.x, xb, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(solve_status, st.status, sizeof(int) * B, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(iterations, st.iterations, sizeof(int) * B, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(violation, st.violation, sizeof(double) * B, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(mu, st.mu, sizeof(double) * B, cudaMemcpyDeviceToHost, s);
    if (status_counts) cudaMemcpyAsync(status_counts, st.counts, sizeof(int) * 4, cudaMemcpyDeviceToHost, s);
    if (loop_count) cudaMemcpyAsync(loop_count, st.loop_count, sizeof(int), cudaMemcpyDeviceToHost, s);
  }
  e = cudaStreamSynchronize(s);
  if (rc != TWB_OK) return rc;
  if (e != cudaSuccess) return CudaFail(e, "solve");
  return TWB_OK;
}

int twb_batch_lm_solve_graph_stats(const twb_batch* b, int* instantiations) {
  if (!b || !instantiations) return Fail(TWB_ERR_INVALID, "null argument");
  *instantiations = b->solve_instantiations;
  return TWB_OK;
}

int twb_batch_lm_solve_radius(const twb_batch* b, double* radius, double* step_norm) {
  if (!b || !radius || !step_norm) return Fail(TWB_ERR_INVALID, "null argument");
  if (!b->lm_radius) return Fail(TWB_ERR_INVALID, "no trust-region solve has run on this batch");
  cudaError_t e = cudaSetDevice(b->device);
  if (e == cudaSuccess) e = cudaStreamSynchronize(b->stream);
  if (e == cudaSuccess) e = cudaMemcpy(radius, b->lm_radius, sizeof(double) * b->B, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(step_norm, b->lm_radius + b->B, sizeof(double) * b->B, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return CudaFail(e, "radius copy");
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
  for (size_t c = 0; c < n_chunks; ++c) {
    const size_t off = c * chunk, nb = std::min(chunk, B - off), tile0 = off / 32;
    if ((e = cudaMemcpyAsync(b->d_x + off * f.n, x + off * f.n, sizeof(double) * nb * f.n, cudaMemcpyHostToDevice, b->s_in)) != cudaSuccess)
      return CudaFail(e, "H2D copy");
    cudaEventRecord(b->ev_chunk[2 * c], b->s_in);
    cudaStreamWaitEvent(s, b->ev_chunk[2 * c], 0);
    int rc = twb::LaunchEval(b->plan, b->d_x + off * f.n, b->d_XT + tile0 * (size_t)(f.n + 1) * 32,
                             b->d_FS ? b->d_FS + tile0 * (size_t)b->plan.n_dyn * 6 * b->plan.n_ee * 32 : nullptr,
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
