// towr_b200_ifopt.hpp — header-only C++ host layer above the C ABI (towr_b200.h) that mirrors, for the NLP
// evaluation path, the interfaces the reference hands to IPOPT:
//
//   * the ifopt Component API — Component / VariableSet / ConstraintSet / CostTerm with GetValues, GetBounds,
//     GetRows, GetName, FillJacobianBlock(var_set, Jacobian&) — as used by every towr constraint class
//     (towr/include/towr/constraints/*.h, e.g. dynamic_constraint.h:62-103, and nodes_variables.h:33), and
//   * towr::NlpFormulation's public fields (towr/include/towr/nlp_formulation.h:100-105) with
//     GetVariableSets / GetConstraints / GetCosts (nlp_formulation.cc:63-376),
//
// served for batch index `b` of a twb_batch from the result of the last batched evaluation.  ifopt and Eigen are
// not available in this image, so ifopt 2.0's classes are restated here in namespace twb_ifopt with the same
// signatures — Component {GetValues, GetBounds, SetVariables, GetJacobian, GetRows, GetName, Print, SetRows,
// kSpecifyLater}, Composite, VariableSet, ConstraintSet {LinkWithVariables, GetJacobian final, FillJacobianBlock,
// InitVariableDependedQuantities}, CostTerm {GetCost} — over two small stand-ins for Eigen::VectorXd and
// Eigen::SparseMatrix<double, RowMajor>.  Nothing here computes: all arithmetic happens in libtowr_b200.so.
#ifndef TOWR_B200_IFOPT_HPP_
#define TOWR_B200_IFOPT_HPP_

#include <algorithm>
#include <array>
#include <cassert>
#include <cstdio>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "towr_b200.h"

// A build that has ifopt includes its headers first and defines TWB_IFOPT_EXTERNAL to its namespace:
//     #include <ifopt/problem.h>
//     #define TWB_IFOPT_EXTERNAL ifopt
//     #include "towr_b200_ifopt.hpp"
// The Gpu* classes below then derive from the real ifopt::VariableSet / ConstraintSet / CostTerm.
// tests/cpp/ifopt_conformance.cc compiles exactly that way against a verbatim restatement of ifopt 2.0's class
// declarations (component.h, variable_set.h, constraint_set.h, cost_term.h, composite.h) to prove the classes are concrete.
#ifndef TWB_IFOPT_EXTERNAL
namespace twb_ifopt {   // mirror of namespace ifopt (ifopt 2.0: component.h, composite.h, variable_set.h, constraint_set.h, cost_term.h, bounds.h)

struct Bounds {                                              // ifopt/bounds.h
  Bounds(double lower = 0.0, double upper = 0.0) : lower_(lower), upper_(upper) {}
  double lower_, upper_;
};
static const double inf = 1.0e20;
static const Bounds NoBound = Bounds(-inf, +inf);
static const Bounds BoundZero = Bounds(0.0, 0.0);
static const Bounds BoundGreaterZero = Bounds(0.0, +inf);
static const Bounds BoundSmallerZero = Bounds(-inf, 0.0);

// Eigen::VectorXd restricted to what this path needs
class VectorXd {
 public:
  VectorXd() = default;
  explicit VectorXd(int n) : v_(n, 0.0) {}
  VectorXd(const double* first, const double* last) : v_(first, last) {}
  VectorXd(std::initializer_list<double> l) : v_(l) {}
  static VectorXd Zero(int n) { return VectorXd(n); }
  int size() const { return (int)v_.size(); }
  int rows() const { return (int)v_.size(); }
  double& operator()(int i) { return v_[i]; }
  double operator()(int i) const { return v_[i]; }
  double& operator[](int i) { return v_[i]; }
  double operator[](int i) const { return v_[i]; }
  double* data() { return v_.data(); }
  const double* data() const { return v_.data(); }
  std::vector<double>::const_iterator begin() const { return v_.begin(); }
  std::vector<double>::const_iterator end() const { return v_.end(); }
 private:
  std::vector<double> v_;
};

// Eigen::SparseMatrix<double, Eigen::RowMajor> restricted to what FillJacobianBlock implementations use
class Jacobian {
 public:
  Jacobian(int rows = 0, int cols = 0) : rows_(rows), cols_(cols) {}
  double& coeffRef(int r, int c) { return v_[{r, c}]; }
  int rows() const { return rows_; }
  int cols() const { return cols_; }
  int nonZeros() const { return (int)v_.size(); }
  const std::map<std::pair<int, int>, double>& entries() const { return v_; }   // row-major, ascending column
 private:
  int rows_, cols_;
  std::map<std::pair<int, int>, double> v_;
};

class Component {                                            // ifopt/composite.h: class Component
 public:
  using Ptr = std::shared_ptr<Component>;
  using Jacobian = twb_ifopt::Jacobian;
  using VectorXd = twb_ifopt::VectorXd;
  using VecBound = std::vector<Bounds>;
  Component(int num_rows, const std::string& name) : num_rows_(num_rows), name_(name) {}
  virtual ~Component() = default;
  virtual VectorXd GetValues() const = 0;
  virtual VecBound GetBounds() const = 0;
  virtual void SetVariables(const VectorXd& x) = 0;
  virtual Jacobian GetJacobian() const = 0;
  int GetRows() const { return num_rows_; }
  std::string GetName() const { return name_; }
  virtual void Print(double tolerance, int& index_start) const {
    (void)tolerance;
    std::printf("%-24s %6d rows  [%d .. %d)\n", name_.c_str(), num_rows_, index_start, index_start + num_rows_);
    index_start += num_rows_;
  }
  void SetRows(int num_rows) { num_rows_ = num_rows; }
  static const int kSpecifyLater = -1;
 private:
  int num_rows_ = kSpecifyLater;
  std::string name_;
};

class Composite : public Component {                         // ifopt/composite.h: class Composite
 public:
  using Ptr = std::shared_ptr<Composite>;
  using ComponentVec = std::vector<Component::Ptr>;
  Composite(const std::string& name, bool is_cost) : Component(0, name), is_cost_(is_cost) {}
  virtual ~Composite() = default;
  VectorXd GetValues() const override {
    VectorXd g_all(GetRows());
    int row = 0;
    for (const auto& c : components_) {
      const VectorXd g = c->GetValues();
      for (int i = 0; i < c->GetRows(); ++i) g_all(row + i) += g(i);
      if (!is_cost_) row += c->GetRows();
    }
    return g_all;
  }
  Jacobian GetJacobian() const override { throw std::runtime_error("Composite::GetJacobian: ask the constraint sets"); }
  VecBound GetBounds() const override {
    VecBound b;
    for (const auto& c : components_) { VecBound bc = c->GetBounds(); b.insert(b.end(), bc.begin(), bc.end()); }
    return b;
  }
  void SetVariables(const VectorXd& x) override {
    int row = 0;
    for (auto& c : components_) {
      VectorXd part(x.data() + row, x.data() + row + c->GetRows());
      c->SetVariables(part);
      row += c->GetRows();
    }
  }
  void PrintAll() const { int i = 0; for (const auto& c : components_) c->Print(0.001, i); }
  const Component::Ptr GetComponent(std::string name) const {
    for (const auto& c : components_) if (c->GetName() == name) return c;
    throw std::runtime_error("component \"" + name + "\" doesn't exist.");
  }
  template <typename T> std::shared_ptr<T> GetComponent(const std::string& name) const {
    std::shared_ptr<T> t = std::dynamic_pointer_cast<T>(GetComponent(name));
    if (!t) throw std::runtime_error("Error casting component " + name);
    return t;
  }
  void AddComponent(const Component::Ptr& c) {
    components_.push_back(c);
    if (is_cost_) SetRows(1); else SetRows(GetRows() + c->GetRows());
  }
  void ClearComponents() { components_.clear(); SetRows(0); }
  const ComponentVec GetComponents() const { return components_; }
 private:
  ComponentVec components_;
  bool is_cost_;
};

class VariableSet : public Component {                       // ifopt/variable_set.h
 public:
  VariableSet(int n_var, const std::string& name) : Component(n_var, name) {}
  virtual ~VariableSet() = default;
  Jacobian GetJacobian() const final { throw std::runtime_error("not implemented for variables"); }
};

class ConstraintSet : public Component {                     // ifopt/constraint_set.h
 public:
  using Ptr = std::shared_ptr<ConstraintSet>;
  using VariablesPtr = Composite::Ptr;
  ConstraintSet(int n_constraints, const std::string& name) : Component(n_constraints, name) {}
  virtual ~ConstraintSet() = default;
  void LinkWithVariables(const VariablesPtr& x) { variables_ = x; InitVariableDependedQuantities(x); }
  // one block per variable set, side by side (constraint_set.cc: GetJacobian)
  Jacobian GetJacobian() const final {
    int n = 0; for (const auto& v : variables_->GetComponents()) n += v->GetRows();
    Jacobian jacobian(GetRows(), n);
    int col = 0;
    for (const auto& v : variables_->GetComponents()) {
      Jacobian jac(GetRows(), v->GetRows());
      FillJacobianBlock(v->GetName(), jac);
      for (const auto& kv : jac.entries()) jacobian.coeffRef(kv.first.first, col + kv.first.second) = kv.second;
      col += v->GetRows();
    }
    return jacobian;
  }
  virtual void FillJacobianBlock(std::string var_set, Jacobian& jac_block) const = 0;
 protected:
  const VariablesPtr GetVariables() const { return variables_; }
 private:
  VariablesPtr variables_;
  virtual void InitVariableDependedQuantities(const VariablesPtr& x_init) { (void)x_init; }
  void SetVariables(const VectorXd& x) final { (void)x; assert(false); }
};

class CostTerm : public ConstraintSet {                      // ifopt/cost_term.h
 public:
  CostTerm(const std::string& name) : ConstraintSet(1, name) {}
  virtual ~CostTerm() = default;
 private:
  virtual double GetCost() const = 0;
 public:
  VectorXd GetValues() const final { VectorXd cost(1); cost(0) = GetCost(); return cost; }
  VecBound GetBounds() const final { return VecBound(GetRows(), NoBound); }
  void Print(double tol, int& index) const final { (void)tol; std::printf("%-24s cost %.6g\n", GetName().c_str(), GetCost()); (void)index; }
};

}  // namespace twb_ifopt
#define TWB_IFOPT_NS twb_ifopt
#else
#define TWB_IFOPT_NS TWB_IFOPT_EXTERNAL
#endif

namespace towr_b200 {

inline void Check(int rc, const char* what) {
  if (rc != TWB_OK) throw std::runtime_error(std::string(what) + ": " + twb_last_error());
}

// B instances of one structure class; stands where B ifopt::Problem objects stand.  Host buffers are plain
// vectors here; a production driver would allocate them pinned (cudaHostAlloc) so the copies overlap.
class BatchedProblem {
 public:
  BatchedProblem(const twb_spec& spec, int batch_size, int device = 0, bool create_batch = true) : B_(batch_size) {
    Check(twb_problem_create(&spec, &prob_), "twb_problem_create");
    Check(twb_problem_dims(prob_, &n_, &m_, &nnz_), "twb_problem_dims");
    row_ptr_.resize(m_ + 1); iRow_.resize(nnz_); jCol_.resize(nnz_);
    Check(twb_problem_row_ptr(prob_, row_ptr_.data()), "twb_problem_row_ptr");
    Check(twb_problem_structure(prob_, iRow_.data(), jCol_.data()), "twb_problem_structure");
    xl_.resize(n_); xu_.resize(n_); gl_.resize(m_); gu_.resize(m_);
    Check(twb_problem_bounds(prob_, xl_.data(), xu_.data(), gl_.data(), gu_.data()), "twb_problem_bounds");
    X.assign((size_t)B_ * n_, 0.0); G.assign((size_t)B_ * m_, 0.0); JAC.assign((size_t)B_ * nnz_, 0.0);
    COST.assign(B_, 0.0); GRAD.assign((size_t)B_ * n_, 0.0); STATUS.assign(B_, 0);
    std::vector<double> x0(n_);
    Check(twb_problem_x0(prob_, x0.data()), "twb_problem_x0");
    for (int b = 0; b < B_; ++b) std::copy(x0.begin(), x0.end(), X.begin() + (size_t)b * n_);
    if (create_batch) Check(twb_batch_create(prob_, B_, device, &batch_), "twb_batch_create");   // TWB_ERR_NO_DEVICE without a GPU
  }
  ~BatchedProblem() { twb_batch_destroy(batch_); twb_problem_destroy(prob_); }
  BatchedProblem(const BatchedProblem&) = delete;
  BatchedProblem& operator=(const BatchedProblem&) = delete;

  // ifopt::Problem::SetVariables(const double*) for instance b
  void SetVariables(int b, const double* x) { std::copy(x, x + n_, X.begin() + (size_t)b * n_); dirty_ = true; }
  // Per-instance start and goal states (what the reference sets in NlpFormulation::initial_base_, final_base_ and
  // initial_ee_W_ before building each request's ifopt::Problem): states[n_states][TWB_STATE_DOUBLES] for instances
  // 0 .. n_states - 1.  Row b of X becomes that instance's initial guess, and from now on the views of instance b serve its
  // own variable and constraint bounds (twb_problem_state_instances; host only, so it also works without a device batch).
  // Instances past n_states keep their rows and bounds.
  void SetStates(const double* states, int n_states = -1) {
    if (n_states < 0) n_states = B_;
    if (!states || n_states == 0 || n_states > B_) throw std::runtime_error("BatchedProblem::SetStates: bad argument");
    if (ixl_.empty()) {   // first call: every instance starts from the problem's bounds
      ixl_.resize((size_t)B_ * n_); ixu_.resize((size_t)B_ * n_); igl_.resize((size_t)B_ * m_); igu_.resize((size_t)B_ * m_);
      for (int b = 0; b < B_; ++b) {
        std::copy(xl_.begin(), xl_.end(), ixl_.begin() + (size_t)b * n_); std::copy(xu_.begin(), xu_.end(), ixu_.begin() + (size_t)b * n_);
        std::copy(gl_.begin(), gl_.end(), igl_.begin() + (size_t)b * m_); std::copy(gu_.begin(), gu_.end(), igu_.begin() + (size_t)b * m_);
      }
    }
    Check(twb_problem_state_instances(prob_, n_states, states, X.data(), ixl_.data(), ixu_.data(), igl_.data(), igu_.data()),
          "twb_problem_state_instances");
    dirty_ = true;
  }
  // one batched evaluation: Problem::EvaluateConstraints + EvalNonzerosOfJacobian + EvaluateCostFunction[Gradient]
  void Evaluate(unsigned flags = TWB_EVAL_ALL) {
    if (!batch_) throw std::runtime_error("BatchedProblem: no device batch");
    Check(twb_batch_eval_host(batch_, X.data(), G.data(), JAC.data(), COST.data(), GRAD.data(), STATUS.data(), flags), "twb_batch_eval_host");
    if (flags == TWB_EVAL_ALL) dirty_ = false;
  }
  // The views evaluate lazily: a SetVariables on any view marks the batch dirty, the next Get* of a constraint / cost view
  // runs ONE batched evaluation for all instances (a lock-step driver sets all iterates first).  Without a device batch
  // (structure-only use) the host arrays are served as they are.
  void MarkDirty() { dirty_ = true; }
  void EnsureEvaluated() { if (dirty_ && batch_) Evaluate(TWB_EVAL_ALL); }
  // ipopt.Solve(nlp) for every instance at once (hopper_example.cc:93): the device-side solve loop of twb_batch_lm_solve_device
  // from the current X, against each instance's own bounds after SetStates (else the problem's), through its host twin
  // twb_batch_lm_solve_host (this header needs no CUDA runtime).  X receives the solutions, so GpuProblem(*this, b)
  // .GetVariableValues() returns instance b's; the constraint and cost views re-evaluate at them on their next Get*.
  // solve_status(b), solve_iterations(b) and solve_violation(b) report per instance.  Returns the call's TWB_* code
  // (TWB_ERR_NO_DEVICE without a device batch; twb_last_error() says more).
  int Solve(const twb_lm_solve_options& opt) {
    if (!batch_) return TWB_ERR_NO_DEVICE;
    SOLVE_STATUS.assign(B_, 0); SOLVE_ITERATIONS.assign(B_, 0); SOLVE_VIOLATION.assign(B_, 0.0); SOLVE_MU.assign(B_, 0.0);
    const bool own = !ixl_.empty();
    const int rc = twb_batch_lm_solve_host(batch_, X.data(), own ? ixl_.data() : nullptr, own ? ixu_.data() : nullptr, own ? igl_.data() : nullptr,
                                           own ? igu_.data() : nullptr, &opt, SOLVE_STATUS.data(), SOLVE_ITERATIONS.data(), SOLVE_VIOLATION.data(),
                                           SOLVE_MU.data(), nullptr, nullptr);
    if (rc == TWB_OK) dirty_ = true;
    return rc;
  }
  int solve_status(int b) const { return SOLVE_STATUS.at(b); }         // TWB_LM_* of the last Solve
  int solve_iterations(int b) const { return SOLVE_ITERATIONS.at(b); } // trials taken
  double solve_violation(int b) const { return SOLVE_VIOLATION.at(b); }   // max |s r| at the returned x
  // ---- solution post-processing of the current X (fpowr) ----
  // fpowr::GetTrajectory(solution, dt) for every instance: [B][n_samples][19 + 13 n_ee]
  std::vector<double> SampleTrajectory(double dt, int* n_samples = nullptr, int* n_values = nullptr) {
    if (!batch_) throw std::runtime_error("BatchedProblem: no device batch");
    int ns = 0, nv = 0;
    Check(twb_problem_trajectory_dims(prob_, dt, &ns, &nv), "twb_problem_trajectory_dims");
    std::vector<double> out((size_t)B_ * ns * nv);
    Check(twb_batch_sample_trajectory_host(batch_, X.data(), dt, out.data()), "twb_batch_sample_trajectory_host");
    if (n_samples) *n_samples = ns;
    if (n_values) *n_values = nv;
    return out;
  }
  // fpowr::ExtractInitialGuesses at the given sample times: [B][times.size()][49] = time | state[12] | controls[36]
  std::vector<double> ExtractInitialGuesses(const std::vector<double>& times) {
    if (!batch_) throw std::runtime_error("BatchedProblem: no device batch");
    std::vector<double> out((size_t)B_ * times.size() * 49);
    Check(twb_batch_initial_guess_host(batch_, X.data(), times.data(), (int)times.size(), out.data()), "twb_batch_initial_guess_host");
    return out;
  }
  // fpowr::ExtractFootstepPlan without the plane lookup: [B][max_states][2 + 4 n_ee], n_states[b] footstep states each
  std::vector<double> ExtractFootstepPlans(double time_horizon, std::vector<int>* n_states, int* max_states = nullptr, int* n_values = nullptr) {
    if (!batch_) throw std::runtime_error("BatchedProblem: no device batch");
    int ms = 0, nv = 0;
    Check(twb_problem_footstep_plan_dims(prob_, &ms, &nv), "twb_problem_footstep_plan_dims");
    std::vector<double> out((size_t)B_ * ms * nv);
    n_states->assign(B_, 0);
    Check(twb_batch_footstep_plan_host(batch_, X.data(), time_horizon, n_states->data(), out.data()), "twb_batch_footstep_plan_host");
    if (max_states) *max_states = ms;
    if (n_values) *n_values = nv;
    return out;
  }
  int GetNumberOfOptimizationVariables() const { return n_; }
  int GetNumberOfConstraints() const { return m_; }
  int nnz() const { return nnz_; }
  int batch_size() const { return B_; }
  const std::vector<int>& row_ptr() const { return row_ptr_; }
  const std::vector<int>& jCol() const { return jCol_; }
  const std::vector<int>& iRow() const { return iRow_; }
  const std::vector<double>& x_lower() const { return xl_; }
  const std::vector<double>& x_upper() const { return xu_; }
  const std::vector<double>& g_lower() const { return gl_; }
  const std::vector<double>& g_upper() const { return gu_; }
  // instance b's bounds: the problem's (the accessors above) until SetStates gives the instance its own
  const double* x_lower(int b) const { return ixl_.empty() ? xl_.data() : ixl_.data() + (size_t)b * n_; }
  const double* x_upper(int b) const { return ixu_.empty() ? xu_.data() : ixu_.data() + (size_t)b * n_; }
  const double* g_lower(int b) const { return igl_.empty() ? gl_.data() : igl_.data() + (size_t)b * m_; }
  const double* g_upper(int b) const { return igu_.empty() ? gu_.data() : igu_.data() + (size_t)b * m_; }
  const twb_problem* handle() const { return prob_; }

  std::vector<double> X, G, JAC, COST, GRAD;   // [B][n], [B][m], [B][nnz], [B], [B][n]
  std::vector<int> STATUS;
  std::vector<int> SOLVE_STATUS, SOLVE_ITERATIONS;   // [B] each, from the last Solve
  std::vector<double> SOLVE_VIOLATION, SOLVE_MU;     // [B] each, from the last Solve

 private:
  twb_problem* prob_ = nullptr;
  twb_batch* batch_ = nullptr;
  int B_, n_ = 0, m_ = 0, nnz_ = 0;
  bool dirty_ = false;
  std::vector<int> row_ptr_, iRow_, jCol_;
  std::vector<double> xl_, xu_, gl_, gu_;
  std::vector<double> ixl_, ixu_, igl_, igu_;   // [B][n], [B][n], [B][m], [B][m] after SetStates, else empty
};

namespace ifo = TWB_IFOPT_NS;

// "base-lin", "ee-motion_0", "ee-schedule1", ... (NodesVariables / PhaseDurations, nodes_variables.cc:40-72,
// phase_durations.cc:68-110) of instance b: a window of row b of X, bounded by instance b's variable bounds
class GpuVariableSet : public ifo::VariableSet {
 public:
  GpuVariableSet(BatchedProblem* p, int b, const std::string& name, int col0, int n) : VariableSet(n, name), p_(p), b_(b), col0_(col0) {}
  VectorXd GetValues() const override {
    VectorXd v(GetRows());
    const double* x = p_->X.data() + (size_t)b_ * p_->GetNumberOfOptimizationVariables() + col0_;
    for (int i = 0; i < GetRows(); ++i) v(i) = x[i];
    return v;
  }
  VecBound GetBounds() const override {
    VecBound v;
    const double *lo = p_->x_lower(b_), *up = p_->x_upper(b_);
    for (int i = 0; i < GetRows(); ++i) v.push_back(ifo::Bounds(lo[col0_ + i], up[col0_ + i]));
    return v;
  }
  // NodesVariables::SetVariables (nodes_variables.cc:65-72): the values move into the batch's iterate; the next Get* of a
  // constraint or cost view re-evaluates the batch
  void SetVariables(const VectorXd& x) override {
    double* dst = p_->X.data() + (size_t)b_ * p_->GetNumberOfOptimizationVariables() + col0_;
    for (int i = 0; i < GetRows(); ++i) dst[i] = x(i);
    p_->MarkDirty();
  }
  int col0() const { return col0_; }
 private:
  BatchedProblem* p_; int b_, col0_;
};

// "dynamic", "rangeofmotion-0", "terrain-ee-motion_0", ... (towr::DynamicConstraint etc.) of instance b, with instance b's
// constraint bounds
class GpuConstraintSet : public ifo::ConstraintSet {
 public:
  GpuConstraintSet(BatchedProblem* p, int b, const std::string& name, int row0, int rows,
                   std::map<std::string, std::pair<int, int>> var_cols)
      : ConstraintSet(rows, name), p_(p), b_(b), row0_(row0), var_cols_(std::move(var_cols)) {}
  VectorXd GetValues() const override {
    p_->EnsureEvaluated();
    VectorXd v(GetRows());
    const double* g = p_->G.data() + (size_t)b_ * p_->GetNumberOfConstraints() + row0_;
    for (int i = 0; i < GetRows(); ++i) v(i) = g[i];
    return v;
  }
  VecBound GetBounds() const override {
    VecBound v;
    const double *lo = p_->g_lower(b_), *up = p_->g_upper(b_);
    for (int i = 0; i < GetRows(); ++i) v.push_back(ifo::Bounds(lo[row0_ + i], up[row0_ + i]));
    return v;
  }
  // the (rows x n_var_set) block of this set's Jacobian w.r.t. one variable set: a slice of the CSR value array
  void FillJacobianBlock(std::string var_set, Jacobian& jac) const override {
    auto it = var_cols_.find(var_set);
    if (it == var_cols_.end()) return;
    p_->EnsureEvaluated();
    const int c0 = it->second.first, nc = it->second.second;
    const double* v = p_->JAC.data() + (size_t)b_ * p_->nnz();
    for (int r = 0; r < GetRows(); ++r)
      for (int k = p_->row_ptr()[row0_ + r]; k < p_->row_ptr()[row0_ + r + 1]; ++k) {
        const int c = p_->jCol()[k];
        if (c0 <= c && c < c0 + nc) jac.coeffRef(r, c - c0) = v[k];
      }
  }
 private:
  // the reference's constraints fetch their variable sets here (e.g. force_constraint.cc:51-60); the views need nothing
  void InitVariableDependedQuantities(const VariablesPtr& x_init) override { (void)x_init; }
  BatchedProblem* p_; int b_, row0_;
  std::map<std::string, std::pair<int, int>> var_cols_;
};

// the summed NodeCost terms of instance b (ifopt sums all cost terms into one row; node_cost.cc:53-76)
class GpuCostTerm : public ifo::CostTerm {
 public:
  GpuCostTerm(BatchedProblem* p, int b, std::map<std::string, std::pair<int, int>> var_cols) : CostTerm("cost"), p_(p), b_(b), var_cols_(std::move(var_cols)) {}
  double Cost() const { return GetCost(); }
  // NodeCost::FillJacobianBlock (node_cost.cc:65-76): the gradient entries of one variable set
  void FillJacobianBlock(std::string var_set, Jacobian& jac) const override {
    auto it = var_cols_.find(var_set);
    if (it == var_cols_.end()) return;
    p_->EnsureEvaluated();
    const double* gr = GetGradient();
    for (int c = 0; c < it->second.second; ++c) if (gr[it->second.first + c] != 0.0) jac.coeffRef(0, c) = gr[it->second.first + c];
  }
  const double* GetGradient() const { p_->EnsureEvaluated(); return p_->GRAD.data() + (size_t)b_ * p_->GetNumberOfOptimizationVariables(); }
 private:
  double GetCost() const override { p_->EnsureEvaluated(); return p_->COST[b_]; }
  BatchedProblem* p_; int b_;
  std::map<std::string, std::pair<int, int>> var_cols_;
};

// towr::NlpFormulation: same public fields; GetVariableSets / GetConstraints / GetCosts return the GPU-backed views
struct State3 { double p[3] = {0, 0, 0}, v[3] = {0, 0, 0}; };
struct BaseState { State3 lin, ang; };
class NlpFormulation {
 public:
  using VariablePtrVec = std::vector<std::shared_ptr<ifo::VariableSet>>;     // nlp_formulation.h:76-78
  using ConstraintPtrVec = std::vector<std::shared_ptr<ifo::ConstraintSet>>;
  using CostPtrVec = std::vector<std::shared_ptr<ifo::CostTerm>>;

  explicit NlpFormulation(int robot = TWB_MONOPED, int terrain = TWB_FLAT) { Check(twb_spec_default(&params_, robot), "twb_spec_default"); params_.terrain = terrain; }

  BaseState initial_base_, final_base_;             // nlp_formulation.h:100-101
  std::vector<std::array<double, 3>> initial_ee_W_; // :102
  twb_spec params_;                                 // towr::Parameters + model_ + terrain_ (:103-105)

  // GaitGenerator::SetCombo + GetPhaseDurations / IsInContactAtStart for every foot
  void SetGait(int n_ee, int combo, double t_total) { Check(twb_spec_set_gait(&params_, n_ee, combo, t_total), "twb_spec_set_gait"); }
  void OptimizePhaseDurations() { Check(twb_spec_optimize_phase_durations(&params_), "twb_spec_optimize_phase_durations"); }

  twb_spec ToSpec() const {
    twb_spec s = params_;
    for (int k = 0; k < 3; ++k) {
      s.initial_base_lin_pos[k] = initial_base_.lin.p[k]; s.initial_base_lin_vel[k] = initial_base_.lin.v[k];
      s.initial_base_ang_pos[k] = initial_base_.ang.p[k]; s.initial_base_ang_vel[k] = initial_base_.ang.v[k];
      s.final_base_lin_pos[k] = final_base_.lin.p[k]; s.final_base_lin_vel[k] = final_base_.lin.v[k];
      s.final_base_ang_pos[k] = final_base_.ang.p[k]; s.final_base_ang_vel[k] = final_base_.ang.v[k];
    }
    if ((int)initial_ee_W_.size() != s.n_ee) throw std::runtime_error("initial_ee_W_ / ee_in_contact_at_start_ size mismatch");
    for (int e = 0; e < s.n_ee; ++e) for (int k = 0; k < 3; ++k) s.initial_ee_W[e][k] = initial_ee_W_[e][k];
    return s;
  }
  static std::map<std::string, std::pair<int, int>> VariableColumns(const BatchedProblem& p) {
    std::map<std::string, std::pair<int, int>> cols; char name[64]; int a0, na;
    for (int i = 0; i < twb_layout_num_variable_sets(p.handle()); ++i) {
      Check(twb_layout_variable_set(p.handle(), i, name, 64, &a0, &na), "twb_layout_variable_set");
      cols[name] = {a0, na};
    }
    return cols;
  }
  static VariablePtrVec GetVariableSets(BatchedProblem& p, int b) {
    VariablePtrVec v; char name[64]; int c0, nc;
    for (int i = 0; i < twb_layout_num_variable_sets(p.handle()); ++i) {
      Check(twb_layout_variable_set(p.handle(), i, name, 64, &c0, &nc), "twb_layout_variable_set");
      v.push_back(std::make_shared<GpuVariableSet>(&p, b, name, c0, nc));
    }
    return v;
  }
  static ConstraintPtrVec GetConstraints(BatchedProblem& p, int b) {
    const auto cols = VariableColumns(p);
    ConstraintPtrVec v; char name[64]; int a0, na;
    for (int i = 0; i < twb_layout_num_constraint_sets(p.handle()); ++i) {
      Check(twb_layout_constraint_set(p.handle(), i, name, 64, &a0, &na), "twb_layout_constraint_set");
      v.push_back(std::make_shared<GpuConstraintSet>(&p, b, name, a0, na, cols));
    }
    return v;
  }
  static CostPtrVec GetCosts(BatchedProblem& p, int b) { return {std::make_shared<GpuCostTerm>(&p, b, VariableColumns(p))}; }
};

// ifopt::Problem (ifopt/problem.h) for instance b of a batch, assembled the way towr/test/hopper_example.cc:70-75 does
// (AddVariableSet / AddConstraintSet / AddCostSet of everything the formulation returns) and offering what
// IpoptAdapter (Ipopt::TNLP) calls.  Every Evaluate* first moves x into the batch (SetVariables) — the batched
// evaluation behind it runs once per new iterate, for all instances of the batch.
class GpuProblem {
 public:
  using VectorXd = ifo::Component::VectorXd;
  using VecBound = ifo::Component::VecBound;
  using Jacobian = ifo::Component::Jacobian;
  GpuProblem(BatchedProblem& p, int b)
      : p_(&p), b_(b), variables_(std::make_shared<ifo::Composite>("variable-sets", false)), constraints_("constraint-sets", false), costs_("cost-terms", true) {
    for (auto& v : NlpFormulation::GetVariableSets(p, b)) AddVariableSet(v);
    for (auto& c : NlpFormulation::GetConstraints(p, b)) AddConstraintSet(c);
    for (auto& c : NlpFormulation::GetCosts(p, b)) AddCostSet(c);
  }
  void AddVariableSet(std::shared_ptr<ifo::VariableSet> variable_set) { variables_->AddComponent(variable_set); }
  void AddConstraintSet(std::shared_ptr<ifo::ConstraintSet> constraint_set) { constraint_set->LinkWithVariables(variables_); constraints_.AddComponent(constraint_set); }
  void AddCostSet(std::shared_ptr<ifo::CostTerm> cost_set) { cost_set->LinkWithVariables(variables_); costs_.AddComponent(cost_set); }
  void SetVariables(const double* x) { p_->SetVariables(b_, x); }
  int GetNumberOfOptimizationVariables() const { return variables_->GetRows(); }
  int GetNumberOfConstraints() const { return constraints_.GetRows(); }
  bool HasCostTerms() const { return twb_problem_has_cost(p_->handle()) != 0; }
  VecBound GetBoundsOnOptimizationVariables() const { return variables_->GetBounds(); }
  VecBound GetBoundsOnConstraints() const { return constraints_.GetBounds(); }
  VectorXd GetVariableValues() const { return variables_->GetValues(); }
  double EvaluateCostFunction(const double* x) { SetVariables(x); p_->EnsureEvaluated(); return p_->COST[b_]; }
  VectorXd EvaluateCostFunctionGradient(const double* x) {
    SetVariables(x); p_->EnsureEvaluated();
    VectorXd g(p_->GetNumberOfOptimizationVariables());
    for (int i = 0; i < g.size(); ++i) g(i) = p_->GRAD[(size_t)b_ * p_->GetNumberOfOptimizationVariables() + i];
    return g;
  }
  VectorXd EvaluateConstraints(const double* x) { SetVariables(x); return constraints_.GetValues(); }
  // values in the order of the structure IPOPT was given (row-major, ascending column): the CSR value array itself
  void EvalNonzerosOfJacobian(const double* x, double* values) {
    SetVariables(x); p_->EnsureEvaluated();
    std::copy(p_->JAC.begin() + (size_t)b_ * p_->nnz(), p_->JAC.begin() + (size_t)(b_ + 1) * p_->nnz(), values);
  }
  // the sparsity structure (Problem::GetJacobianOfConstraints as IpoptAdapter::eval_jac_g reads it)
  const std::vector<int>& GetJacobianRows() const { return p_->iRow(); }
  const std::vector<int>& GetJacobianCols() const { return p_->jCol(); }
  Jacobian GetJacobianOfConstraints() const {
    p_->EnsureEvaluated();
    Jacobian jac(p_->GetNumberOfConstraints(), p_->GetNumberOfOptimizationVariables());
    const double* v = p_->JAC.data() + (size_t)b_ * p_->nnz();
    for (int k = 0; k < p_->nnz(); ++k) jac.coeffRef(p_->iRow()[k], p_->jCol()[k]) = v[k];
    return jac;
  }
  const ifo::Composite& GetConstraints() const { return constraints_; }
  const ifo::Composite& GetCosts() const { return costs_; }
  ifo::Composite::Ptr GetOptVariables() const { return variables_; }
  void PrintCurrent() const { variables_->PrintAll(); constraints_.PrintAll(); costs_.PrintAll(); }
 private:
  BatchedProblem* p_; int b_;
  ifo::Composite::Ptr variables_;
  ifo::Composite constraints_, costs_;
};

}  // namespace towr_b200
#endif  // TOWR_B200_IFOPT_HPP_
