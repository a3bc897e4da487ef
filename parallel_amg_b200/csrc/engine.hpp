// engine.hpp — device engine interface used by the C ABI (capi.cpp).  No CUDA types leak out.
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "host.hpp"

typedef struct CUgraphExec_st* cudaGraphExec_t;

namespace pamg {

struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
struct NoGpuError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
struct CommError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

struct OpSpec;
struct EpiArgs;
struct PartDev;

enum VecId { V_X = 0, V_X2, V_B, V_T, V_XSTART, V_XSOL, V_P, V_Q, V_BSAVE };

class Engine {
 public:
  // kmax: columns of per-solve device state (right-hand sides a multi-column call may use), 1..PAMG_MAX_RHS
  Engine(Hierarchy* h, int nlocal, const int32_t* local_parts, const int32_t* device_ids, int kmax = 1);
  ~Engine();
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;

  static int32_t handle_bytes();
  int rhs_capacity() const;
  void export_handle(int part, void* blob);
  void import_handle(int part, const void* blob);
  void connect();

  void spmv(int level, const double* const* x, double* const* y);
  void consistent(int level, double* const* v);
  void assemble(int level, double* const* v);
  void smooth(int level, int nu, const double* const* b, double* const* x);
  void residual_restrict(int level, const double* const* b, const double* const* x, double* const* r, double* const* bc);
  void prolong_correct(int level, const double* const* ec, double* const* x);
  double dot(int level, const double* const* u, const double* const* v);
  void vcycle(const double* const* b, double* const* x);
  int pcg(const double* const* b, double* const* x, double rtol, int maxiter, int mode, int* iters, double* hist);
  // k right-hand sides: vectors at [j * nparts + part]; column j bit-identical to the single-column call on it
  void spmv_multi(int level, int k, const double* const* x, double* const* y);
  void vcycle_multi(int k, const double* const* b, double* const* x);
  void time_kernel_multi(int k, int kind, int level, int reps, bool flush_l2, float* ms_out);
  int pcg_multi(int k, const double* const* b, double* const* x, double rtol, int maxiter, int mode, int* iters, int* converged,
                double* hist);
  int fgmres(const double* const* b, double* const* x, double rtol, int maxiter, int restart, int precond, int* iters,
             double* hist);
  void load_rhs(const double* const* b);
  int pcg_resident(double rtol, int maxiter, int mode, int* iters, double* hist);
  void read_solution(double* const* x);
  void time_kernel(int kind, int level, int reps, bool flush_l2, float* ms_out);
  void get_stats(pamg_stats* s);
  void trace_enable(int capacity);
  int trace_read(int part, unsigned long long* out, int cap);
  std::string trace_names();

 private:
  struct Impl;
  Impl* impl;

  void plan_buffers();
  void require_connected();
  void sync_all();
  void upload_vec(int level, const double* const* host, int which_buf);
  void download_vec(int level, double* const* host, int which_buf);
  void download_own(PartDev& pd, int level, const double* src, double* host);
  double* vec(PartDev& pd, int level, int which);
  std::vector<const double*> ptrs(int level, int which);
  void check_device_error();
  void clear_done();
  void enqueue_op(const OpSpec& op, const std::vector<const double*>& xin, const std::vector<EpiArgs>& epi);
  void enqueue_smooth(int l, int nu, std::vector<double*>& cur, bool zero_guess_done, bool dot_last);
  void enqueue_tail(bool zero_guess);
  void enqueue_vcycle(int l, bool dot_rz, bool zero_guess);
  void enqueue_vcycle_entry();
  void enqueue_dot_rz();
  bool vcycle_fuses_rz() const;
  void enqueue_pcg_iteration(int mode);
  int run_pcg(double rtol, int maxiter, int mode, int* iters, int* converged, double* hist);
  void begin_multi(int k);
  void end_multi();
  template <class F>
  auto in_multi(int k, F&& body) -> decltype(body());
  template <class F>
  void capture(std::vector<cudaGraphExec_t>& out, int64_t* nodes, F&& body);
  void launch_graphs(const std::vector<cudaGraphExec_t>& gs, int64_t nodes);
};

}  // namespace pamg
