// kernels.cuh — hand-written sm_100a kernels of the AMG-PCG solve phase.
//
// Every per-level operation of SURVEY.md 8(a) is an "SpMV + row epilogue":
//   a1 SpMV            out = A x                       (+ fused dot(dotv, out) for PCG's p.q)
//   a2 smoothing       out = x + w (b - A x)           (+ fused dot(r, z) on level 0)
//   a3 residual        out = b - A x ;  restrict  b_c = R r  (+ fused coarse pre-smooth x_c = w_c b_c)
//   a4 prolong+correct out = x + P e_c
// so one templated kernel family (three storage formats) covers them.  Operators with few distinct values (the three
// BASELINE matrices and their prolongators) run the value-indexed SELL kernels (k_spmv_sell_vi4: int32 column + index
// byte(s) into a dictionary of the original doubles, 5-6 instead of 12 bytes per entry, same bits); stencil operators store no
// column at all (k_spmv_sell_diag: one index byte per (row, offset) slot, the column is row + offset).
//
// Halo exchange (PartitionedArrays mul!: start consistent!(b); c_own = A_oo b_own; wait;
// c_own += A_og b_ghost, SURVEY App. A) is FUSED INTO THE SAME KERNEL as three CTA roles:
//   pack CTAs     (lowest block ids)  store this part's boundary values straight into the neighbour
//                                     GPUs' ghost staging over NVLink peer mappings, then publish an
//                                     epoch flag (release, system scope);
//   boundary CTAs (next block ids)    spin on the local flags (acquire), then compute the boundary rows
//                                     completely: own columns, then ghost columns, then the epilogue.
//                                     They are few, latency-bound and dispatched early, so both the NVLink
//                                     latency and their own run behind the main role's streaming;
//   main CTAs                         all rows of the own-own block; rows that also have ghost columns
//                                     ("boundary rows", marked in `skip`) are computed but not stored.
// Staging buffers are double-buffered by epoch parity; see DESIGN.md "Halo protocol" for why that
// is race-free.  When several parts share one GPU (the PartitionedArrays "debug backend" layout
// used by the single-GPU tests) a kernel must never wait for a later kernel of the same stream, so
// the same three roles run as three launches (k_halo_pack, main, k_boundary): identical row
// arithmetic, identical results.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

namespace pamg {

constexpr int RED_W = 4;  // doubles per all-reduce slot
constexpr int MAX_LEVELS = 16;
constexpr int BLOCK = 256;
constexpr unsigned long long SPIN_TIMEOUT_NS = 20000000000ull;  // default 20 s (env PAMG_SPIN_TIMEOUT_MS): then error + done

enum Mode : int { M_MUL = 0, M_RESID = 1, M_JACOBI = 2, M_ADD = 3, M_RESTRICT = 4, M_CHEB = 5 };

// scalar slots in DevState::sc
enum { SC_RHO_OLD = 0, SC_RHO_NEW = 1, SC_RR0 = 2, SC_RR = 3, SC_RTOL = 4, SC_LAST = 5, SC_COUNT = 8 };

struct CsrView {
  const int32_t* ptr;
  const int32_t* col;
  const double* val;
  const int32_t* rows;  // != nullptr: compressed row list (own-ghost blocks): logical row k -> rows[k]
  int32_t nrows;        // logical rows
};

struct EpiArgs {
  double* out;         // y | r | x_new | x | b_c
  const double* in0;   // b (RESID, JACOBI, CHEB) | x (ADD)
  const double* in1;   // x (JACOBI, CHEB)
  const double* w;     // w/a_ii (JACOBI) | w_c (RESTRICT, out2) | 1/a_ii (CHEB)
  double* out2;        // RESTRICT: x_c = w_c b_c | CHEB: d_new
  const double* aux;   // CHEB: d_old
  const double* dotv;  // DOT: sum dotv[i] * out[i]
  double c1, c2;       // CHEB: d_new = c1 d_old + c2 w (b - s)
};

// mutable per-part device state
struct DevState {
  uint32_t red_epoch;
  uint32_t coarse_epoch;
  uint32_t halo_epoch[MAX_LEVELS];
  uint32_t pack_done[MAX_LEVELS];  // fused launches: epoch whose pack role has finished
  uint32_t asm_epoch[MAX_LEVELS];
  uint32_t ticket[8];
  int32_t done;
  int32_t iters;
  int32_t error;
  int32_t maxiter;
  double sc[SC_COUNT];
  double dot_main;  // split launches: partial of the main launch, completed and published by k_boundary
  uint32_t check_seq;  // k_check executions since k_pcg_init
  unsigned long long spin_timeout_ns;  // cross-GPU waits give up after this long (sets error and done)
  unsigned long long* trace;  // != nullptr: CTA 0 of every kernel appends its start time (globaltimer, ns)
  uint32_t trace_pos, trace_cap;
};

// status record k_check stores straight into pinned host memory (no D2H copy between iterations)
struct HostStat {
  uint32_t seq;  // number of the k_check that wrote this slot (written last)
  int32_t done, error, iters;
};
constexpr int HS_RING = 16;

struct RedPub {  // where this part publishes its all-reduce contribution in part d (incl. itself)
  double* slot[2];
  uint32_t* flag;
};
struct RedCtx {
  const RedPub* pubs;      // [nparts]
  const double* local;     // [2][nparts][RED_W] in this part's arena
  const uint32_t* flags;   // [nparts]
  int32_t nparts;
};

struct SendNbr {  // one neighbour of a halo send
  double* ghost[2];  // peer staging (already offset to this part's first slot), per parity
  uint32_t* flag;    // peer flag for this part
  int32_t offset, count;
};
struct HaloRecv {
  const double* ghost[2];
  const uint32_t* flags;
  int32_t n_nbrs;
};

// boundary rows of one operator: the rows of the own-own block that also have own-ghost entries,
// stored whole: entries [ptr[k], mid[k]) index the own vector, [mid[k], ptr[k+1]) the ghost staging
struct BndView {
  const int32_t* rows;  // [n] own-local row ids
  const int32_t* ptr;   // [n + 1]
  const int32_t* mid;   // [n]
  const int32_t* col;
  const double* val;
  int32_t n, lanes;     // lanes: threads per row (power of two <= 32)
};

// what the pack / boundary roles of a fused launch need (n_pack == n_bnd == 0: plain kernel)
struct FusedHalo {
  int32_t n_pack, n_bnd;    // CTAs per role; the main role gets gridDim.x - n_pack - n_bnd
  int32_t level;            // halo level (epoch / flag index)
  int32_t fixed_parity;     // >= 0: ghost values are already in staging[parity], no wait (coarsest level)
  int32_t fused;            // 1: roles inside one launch (boundary role advances the epoch)
  int32_t bnd_first;        // 1: block ids [pack | boundary | main]; 0: [pack | main | boundary]
  int32_t n_send, n_nbrs;   // pack role
  const double* v;
  const int32_t* send_idx;
  const SendNbr* nbrs;
  BndView B;                // boundary role
  HaloRecv hr;
  const uint8_t* skip;      // [nrows] 1 => boundary row: the main role must not store it (nullptr: none)
};

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// tracing: one timestamp per kernel launch, taken by the first thread of CTA 0 (pamg_trace_*)
__device__ __forceinline__ void trace_mark(DevState* st) {
  if (blockIdx.x == 0 && threadIdx.x == 0 && st->trace) {
    const uint32_t i = atomicAdd(&st->trace_pos, 1u);
    if (i < st->trace_cap) st->trace[i] = globaltimer_ns();
  }
}
// streaming (read-once) 64/32-bit loads that do not pollute L1
__device__ __forceinline__ double ldg_stream(const double* p) { return __ldcs(p); }
__device__ __forceinline__ int32_t ldg_stream(const int32_t* p) { return __ldcs(p); }

// Request a line without tying up a register: the epilogue operands of a row (b, w, ...) are prefetched
// into L1 BEFORE the row's entries are streamed and loaded after the loop, when they hit.  (Holding them
// in registers across the loop costs the SELL kernels their load-level parallelism: 0.49 vs 0.40 ms for
// the 256^3 Jacobi sweep; letting nvcc sink the loads below the loop exposes a full DRAM latency.)
__device__ __forceinline__ void prefetch_l1(const double* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

__device__ __forceinline__ void spin_until(const uint32_t* flag, uint32_t e, DevState* st) {
  if ((int32_t)(ld_acquire_sys(flag) - e) >= 0) return;
  if (*(volatile int32_t*)&st->error) return;  // a wait already timed out: fail fast, the host reports it
  const unsigned long long t0 = globaltimer_ns();
  while ((int32_t)(ld_acquire_sys(flag) - e) < 0) {
    if (*(volatile int32_t*)&st->error) return;
    if (globaltimer_ns() - t0 > st->spin_timeout_ns) {
      st->error = 1;  // reported by the host after the call; `done` turns every later kernel of the solve into a no-op
      st->done = 1;
      __threadfence();
      return;
    }
    __nanosleep(64);
  }
}

__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// one thread: wait until flags[0..n) have all reached epoch e.  The polls are relaxed system-scope loads; once every flag
// is there ONE acquire load closes the wait (LDG.STRONG.SYS + an L1 invalidate).  Everything read behind a wait (ghost
// staging, all-reduce slots, gather buffers) is read with ld.cv, i.e. at L2, and is only issued after the branch on the
// flag value, so it cannot be older than the flag.  Measured alternatives: an ld.acquire.sys per flag serialises n L2
// round trips at the head of every consumer (round 1); a __threadfence_system() after the polls is a MEMBAR.SC.SYS in each
// of several hundred waiting CTAs while the main role streams -- +53 us per iteration on 2 GPUs (profiles/r02).
__device__ __forceinline__ void spin_until_all(const uint32_t* flags, int n, uint32_t e, DevState* st) {
  unsigned long long t0 = 0;
  for (int k = 0; k < n; ++k) {
    while ((int32_t)(ld_relaxed_sys(flags + k) - e) < 0) {
      if (*(volatile int32_t*)&st->error) return;  // a wait already timed out: fail fast, the host reports it
      if (t0 == 0) t0 = globaltimer_ns();
      if (globaltimer_ns() - t0 > st->spin_timeout_ns) {
        st->error = 1;
        st->done = 1;
        __threadfence();
        return;
      }
      __nanosleep(32);
    }
  }
  if (n > 0) (void)ld_acquire_sys(flags);
}

// one thread: wait for every neighbour's flag of this level's current epoch; returns parity
__device__ __forceinline__ int halo_wait(const HaloRecv& hr, uint32_t e, DevState* st) {
  spin_until_all(hr.flags, hr.n_nbrs, e, st);
  return (int)(e & 1u);
}

template <int W>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
  for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, W);
  return v;
}

// deterministic block sum (fixed tree); result valid in thread 0
__device__ __forceinline__ double block_sum(double v) {
  __shared__ double sh[BLOCK / 32];
  v = group_sum<32>(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sh[wid] = v;
  __syncthreads();
  if (wid == 0) {
    v = (lane < BLOCK / 32) ? sh[lane] : 0.0;
    v = group_sum<32>(v);
  }
  return v;
}

// last-block detection: returns true (in every thread of exactly one block) once all blocks of
// the grid have passed; the ticket is reset for the next launch.
__device__ __forceinline__ bool last_block_n(uint32_t* ticket, uint32_t n) {
  __shared__ bool is_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const uint32_t t = atomicAdd(ticket, 1u);
    is_last = (t == n - 1);
    if (is_last) *ticket = 0;
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}
__device__ __forceinline__ bool last_block(uint32_t* ticket) { return last_block_n(ticket, gridDim.x); }

// publish v[0..RED_W) to every part (one thread)
__device__ __forceinline__ void red_publish(DevState* st, const RedCtx& rc, const double* v) {
  const uint32_t e = st->red_epoch + 1u;
  for (int d = 0; d < rc.nparts; ++d) {
    double* s = rc.pubs[d].slot[e & 1u];
#pragma unroll
    for (int k = 0; k < RED_W; ++k) s[k] = v[k];
  }
  __threadfence_system();  // one fence, then relaxed flag stores: a release per flag costs a fence each (8 parts: ~16 us)
  for (int d = 0; d < rc.nparts; ++d) *(volatile uint32_t*)rc.pubs[d].flag = e;
  st->red_epoch = e;
}

// one thread: wait for all parts, sum in ascending part order (deterministic, identical on all parts)
__device__ __forceinline__ void red_consume(DevState* st, const RedCtx& rc, double* v) {
  const uint32_t e = *(volatile uint32_t*)&st->red_epoch;
  spin_until_all(rc.flags, rc.nparts, e, st);
  const double* base = rc.local + (size_t)(e & 1u) * rc.nparts * RED_W;
#pragma unroll
  for (int k = 0; k < RED_W; ++k) v[k] = 0.0;
  for (int d = 0; d < rc.nparts; ++d)
#pragma unroll
    for (int k = 0; k < RED_W; ++k) v[k] += __ldcv(base + d * RED_W + k);
}

// block-level finish of a fused dot: per-block partials -> last block sums them in block order.
// publish: 0 = store the local total in st->dot_main (a k_boundary launch follows and publishes),
//          1 = publish total (+ st->dot_main if add_main) to all parts.
// Returns true in exactly one thread of the grid: thread 0 of the last block, after it has published / stored the total.
__device__ __forceinline__ bool dot_finish(double acc, double* partials, DevState* st, uint32_t* ticket,
                                           const RedCtx& rc, int publish, int add_main, int slot) {
  const double bs = block_sum(acc);
  if (threadIdx.x == 0) partials[blockIdx.x] = bs;
  bool mine = false;
  if (last_block(ticket)) {
    double s = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += BLOCK) s += __ldcv(partials + i);
    s = block_sum(s);
    if (threadIdx.x == 0) {
      if (add_main) s += st->dot_main;
      if (publish) {
        double v[RED_W] = {0.0, 0.0, 0.0, 0.0};
        v[slot] = s;
        red_publish(st, rc, v);
      } else {
        st->dot_main = s;
      }
      mine = true;
    }
  }
  return mine;
}

// ---------------------------------------------------------------------------------------------
// row epilogue shared by every SpMV family and by the boundary role
// ---------------------------------------------------------------------------------------------
template <int MODE>
__device__ __forceinline__ double stream_epilogue(const EpiArgs& a, int row, double s, double e_in0, double e_in1, double e_w,
                                                  double e_aux) {
  double res;
  if (MODE == M_MUL) {
    res = s;
    a.out[row] = res;
  } else if (MODE == M_RESID) {
    res = e_in0 - s;
    a.out[row] = res;
  } else if (MODE == M_JACOBI) {
    res = e_in1 + e_w * (e_in0 - s);
    a.out[row] = res;
  } else if (MODE == M_ADD) {
    res = e_in0 + s;
    a.out[row] = res;
  } else if (MODE == M_RESTRICT) {
    res = s;
    a.out[row] = res;
    if (a.out2) a.out2[row] = e_w * s;
  } else {  // M_CHEB
    const double d = a.c1 * e_aux + a.c2 * (e_w * (e_in0 - s));
    a.out2[row] = d;
    res = e_in1 + d;
    a.out[row] = res;
  }
  return res;
}

// loads the operands, applies the epilogue; DOT: returns dotv[row] * result with dotv read BEFORE the
// stores (a load after the store to `out` cannot be hoisted by the compiler and would sit exposed)
template <int MODE, bool DOT = false>
__device__ __forceinline__ double apply_epilogue(const EpiArgs& a, int row, double s) {
  double e_in0 = 0.0, e_in1 = 0.0, e_w = 0.0, e_aux = 0.0, e_dot = 0.0;
  if (MODE == M_RESID || MODE == M_JACOBI || MODE == M_ADD || MODE == M_CHEB) e_in0 = a.in0[row];
  if (MODE == M_JACOBI || MODE == M_CHEB) e_in1 = a.in1[row];
  if (MODE == M_JACOBI || MODE == M_CHEB || (MODE == M_RESTRICT && a.out2)) e_w = a.w[row];
  if (MODE == M_CHEB && a.aux) e_aux = a.aux[row];
  if (DOT) e_dot = (a.dotv == a.in0 && (MODE == M_JACOBI || MODE == M_RESID)) ? e_in0 : a.dotv[row];
  const double res = stream_epilogue<MODE>(a, row, s, e_in0, e_in1, e_w, e_aux);
  return DOT ? e_dot * res : res;
}

// ---------------------------------------------------------------------------------------------
// halo roles (consistent! fused into the consuming kernel)
// ---------------------------------------------------------------------------------------------
// pack role, CTA `bid` of fh.n_pack: owner -> ghost stores into the neighbours' staging, then flags
__device__ __forceinline__ void pack_role(const FusedHalo& fh, DevState* st, int bid) {
  const uint32_t e = *(volatile uint32_t*)&st->halo_epoch[fh.level] + 1u;
  const int par = (int)(e & 1u);
  for (int k = bid * BLOCK + threadIdx.x; k < fh.n_send; k += fh.n_pack * BLOCK) {
    int nb = 0;
    while (nb + 1 < fh.n_nbrs && k >= fh.nbrs[nb + 1].offset) ++nb;
    fh.nbrs[nb].ghost[par][k - fh.nbrs[nb].offset] = fh.v[fh.send_idx[k]];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();  // this CTA's peer stores (cumulative over the barrier) are visible system-wide
    const uint32_t t = atomicAdd(&st->ticket[1], 1u);
    if (t == (uint32_t)fh.n_pack - 1u) {  // every pack CTA has fenced: publish the epoch to the neighbours
      st->ticket[1] = 0;
      __threadfence_system();
      for (int nb = 0; nb < fh.n_nbrs; ++nb) *(volatile uint32_t*)fh.nbrs[nb].flag = e;
      if (fh.fused)
        *(volatile uint32_t*)&st->pack_done[fh.level] = e;  // the boundary role advances the epoch
      else
        st->halo_epoch[fh.level] = e;
    }
  }
}

// partial row sum over entries [beg, end) strided by `lanes`, four entries in flight per lane
template <bool VOLATILE_X>
__device__ __forceinline__ double row_part(const int32_t* __restrict__ col, const double* __restrict__ val, int beg, int end,
                                           int lane, int lanes, const double* x) {
  double s = 0.0;
  for (int q = beg + lane; q < end; q += 4 * lanes) {
    int c[4];
    double v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int qq = q + u * lanes;
      c[u] = qq < end ? ldg_stream(col + qq) : -1;
      v[u] = qq < end ? ldg_stream(val + qq) : 0.0;
    }
    double xv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) xv[u] = c[u] >= 0 ? (VOLATILE_X ? __ldcv(x + c[u]) : x[c[u]]) : 0.0;
#pragma unroll
    for (int u = 0; u < 4; ++u) s += v[u] * xv[u];
  }
  return s;
}

// boundary role, CTA `bid` of fh.n_bnd: the boundary rows whole -- own-column sum first (it does not
// need the halo, so it runs while the neighbours' values are still in flight), then wait for the
// neighbours' flags, ghost-column sum, epilogue.  Returns this thread's dot contribution.
template <int MODE, bool DOT>
__device__ __forceinline__ double boundary_role(const FusedHalo& fh, const double* __restrict__ x, const EpiArgs& a, DevState* st,
                                                int bid) {
  __shared__ int s_par;
  __shared__ uint32_t s_epoch;
  const BndView& B = fh.B;
  const int lanes = B.lanes;
  const int lane = threadIdx.x & (lanes - 1);
  const int grp = threadIdx.x / lanes;
  const int rpb = BLOCK / lanes;
  bool waited = false;
  const double* g = nullptr;
  auto wait_halo = [&]() {  // block-uniform call sites only
    if (threadIdx.x == 0) {
      if (fh.fixed_parity >= 0) {
        s_par = fh.fixed_parity;
        s_epoch = 0;
      } else {
        const uint32_t e = *(volatile uint32_t*)&st->halo_epoch[fh.level] + (fh.fused ? 1u : 0u);
        s_par = halo_wait(fh.hr, e, st);
        s_epoch = e;
      }
    }
    __syncthreads();
    g = fh.hr.ghost[s_par];
    waited = true;
  };
  double acc = 0.0;
  // block-uniform trip count: every lane reaches the barrier and the full-mask shuffles
  for (int k0 = bid * rpb; k0 < B.n; k0 += fh.n_bnd * rpb) {
    const int k = k0 + grp;
    const bool valid = k < B.n;
    int beg = 0, mid = 0, end = 0;
    if (valid) {
      beg = B.ptr[k];
      mid = B.mid[k];
      end = B.ptr[k + 1];
    }
    double s = row_part<false>(B.col, B.val, beg, mid, lane, lanes, x);
    if (!waited) wait_halo();
    double sg = row_part<true>(B.col, B.val, mid, end, lane, lanes, g);
    for (int o = lanes >> 1; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      sg += __shfl_xor_sync(0xffffffffu, sg, o);
    }
    if (valid && lane == 0) {
      const int row = B.rows[k];
      const double res = apply_epilogue<MODE, DOT>(a, row, s + sg);  // mul!: own-own sum, then += own-ghost sum
      if (DOT) acc += res;
    }
  }
  if (!waited) wait_halo();  // a CTA without rows still consumes the exchange (keeps the epoch protocol in step)
  if (fh.fused && fh.fixed_parity < 0 && last_block_n(&st->ticket[4], (uint32_t)fh.n_bnd)) {
    if (threadIdx.x == 0) {  // every boundary CTA has consumed epoch e: advance once the local pack is out
      const uint32_t e = s_epoch;
      if (fh.n_pack > 0) spin_until(&st->pack_done[fh.level], e, st);
      *(volatile uint32_t*)&st->halo_epoch[fh.level] = e;
    }
  }
  return acc;
}

// ---------------------------------------------------------------------------------------------
// sub-warp CSR ("vector per row") SpMV family: LANES threads per row (32 = warp per row)
// ---------------------------------------------------------------------------------------------
template <int LANES, int MODE, bool DOT>
__global__ void __launch_bounds__(BLOCK) k_spmv(CsrView A, const double* __restrict__ x, EpiArgs a, DevState* st, FusedHalo fh,
                                                 double* partials, RedCtx rc, int publish, int red_slot) {
  if (st->done) return;
  trace_mark(st);
  double acc = 0.0;
  int bid = blockIdx.x;
  const int n_main = (int)gridDim.x - fh.n_pack - fh.n_bnd;
  const int b0 = fh.n_pack + (fh.bnd_first ? 0 : n_main);  // first boundary CTA
  if (bid < fh.n_pack) {
    pack_role(fh, st, bid);
  } else if (bid >= b0 && bid < b0 + fh.n_bnd) {
    acc = boundary_role<MODE, DOT>(fh, x, a, st, bid - b0);
  } else {
    bid -= fh.n_pack + (fh.bnd_first ? fh.n_bnd : 0);
    constexpr int RPB = BLOCK / LANES;
    const int lane = threadIdx.x % LANES;
    const int grp = threadIdx.x / LANES;
    // block-uniform trip count: every lane of a warp reaches the full-mask shuffles below, rows past
    // the end are just predicated off (a lane that skipped the loop would deadlock the shuffle)
    for (int r0 = bid * RPB; r0 < A.nrows; r0 += n_main * RPB) {
      const int r = r0 + grp;
      const bool valid = r < A.nrows;
      int beg = 0, end = 0;
      unsigned char sk = 0;
      if (valid) {
        beg = A.ptr[r];
        end = A.ptr[r + 1];
        if (fh.skip) sk = fh.skip[r];
      }
      double s = 0.0;
      for (int k = beg + lane; k < end; k += LANES) {
        const int c = ldg_stream(A.col + k);
        const double v = ldg_stream(A.val + k);
        s += v * x[c];
      }
      s = group_sum<LANES>(s);
      if (valid && lane == 0 && !sk) {
        const double res = apply_epilogue<MODE, DOT>(a, r, s);
        if (DOT) acc += res;
      }
    }
  }
  if (DOT) dot_finish(acc, partials, st, &st->ticket[0], rc, publish, 0, red_slot);
}

// boundary role as its own launch (several parts on one GPU); completes a dot started by the main launch
template <int MODE, bool DOT>
__global__ void __launch_bounds__(BLOCK) k_boundary(const double* __restrict__ x, EpiArgs a, DevState* st, FusedHalo fh,
                                                     double* partials, RedCtx rc, int red_slot) {
  if (st->done) return;
  trace_mark(st);
  const double acc = boundary_role<MODE, DOT>(fh, x, a, st, blockIdx.x);
  if (DOT) dot_finish(acc, partials, st, &st->ticket[0], rc, 1, 1, red_slot);
}

// ---------------------------------------------------------------------------------------------
// CSR-stream SpMV family (the fast path for the own-own blocks).
//
// The vector kernel above is latency-bound on short rows (ncu, profiles/r01: ~18 % DRAM
// throughput at full occupancy, long-scoreboard stalls: a serial ptr -> col/val -> x chain with
// ~12 B in flight per thread).  Here a CTA owns a run of consecutive rows whose entries fit the
// shared-memory product buffer; the run's val/col ranges are CONTIGUOUS in CSR, so phase A streams
// them with fully coalesced 128-bit loads (int4 of 4 column ids + 2 x double2 of values per thread
// and step, all steps issued back to back: up to 144 B in flight per thread), gathers x through
// L1/L2 and parks the products in shared memory; phase B sums each row's products in column order
// (one thread per row) and applies the fused epilogue, whose operands were prefetched before
// phase A.  Products are rounded before they are added (no FMA across the smem round trip), so a
// row sum is bit-identical to the oracle's sequential `s += a_ij * x_j`.
// ---------------------------------------------------------------------------------------------
constexpr int S_CAP = 3072;        // entries per row block (24 KB of fp64 products)
constexpr int S_CHUNKS = 4;        // phase B handles up to S_CHUNKS rows per thread
constexpr int S_ROWS = S_CHUNKS * BLOCK;  // rows per row block
constexpr int S_STEPS = (S_CAP + 4 * BLOCK - 1) / (4 * BLOCK);
constexpr int RED_GRID = 148 * 8;  // upper bound of the CTAs of a kernel with a fused reduction (one fence + ticket per CTA)

struct StreamView {
  const int2* blk;     // [nblocks + 1] {first row, first entry} of each row block
  const int32_t* ptr;
  const int32_t* col;  // padded with zeros to a multiple of 4 entries (+ 8)
  const double* val;
  int32_t nrows, nblocks;
};

// The grid is the number of row blocks (one block per CTA, hardware-scheduled) except for the
// variants with a fused dot product, which run RED_GRID CTAs that stride over the row blocks: a
// gpu-scope fence per CTA (needed by the last-block reduction) invalidates the SM's L1, so it must
// not happen once per row block (ncu r01: +45 % time with 65536 fencing CTAs).
// LONG (rows of >= 48 entries on average: the restriction operators of the coarse levels, 240 entries per row at 256^3, and
// the Galerkin matrices of the tail): a row block then holds a dozen rows, and one thread per row leaves 244 of 256 threads
// idle through a 240-step dependent add chain (restrict R1: 68 us for 146 MB).  Phase B there gives every row S_LB lanes:
// lane j adds the products k = j, j + S_LB, ... in ascending order, then a fixed xor tree over the lanes: deterministic,
// but not the oracle's left-to-right order (1e-16 relative, like the sub-warp CSR family).
template <int MODE, bool DOT, bool LONG = false>
__global__ void __launch_bounds__(BLOCK, 4) k_spmv_stream(StreamView A, const double* __restrict__ x, EpiArgs a, DevState* st,
                                                        FusedHalo fh, double* partials, RedCtx rc, int publish, int red_slot) {
  if (st->done) return;
  trace_mark(st);
  __shared__ double prod[S_STEPS * 4 * BLOCK];
  const int t = threadIdx.x;
  double acc = 0.0;
  const int n_main = (int)gridDim.x - fh.n_pack - fh.n_bnd;
  int bk0 = (int)blockIdx.x - fh.n_pack - (fh.bnd_first ? fh.n_bnd : 0);
  const int b0 = fh.n_pack + (fh.bnd_first ? 0 : n_main);  // first boundary CTA
  if ((int)blockIdx.x < fh.n_pack) {
    pack_role(fh, st, blockIdx.x);
    bk0 = A.nblocks;  // no main work
  } else if ((int)blockIdx.x >= b0 && (int)blockIdx.x < b0 + fh.n_bnd) {
    acc = boundary_role<MODE, DOT>(fh, x, a, st, (int)blockIdx.x - b0);
    bk0 = A.nblocks;
  }
  for (int bk = bk0; bk < A.nblocks; bk += n_main) {
    const int2 b0 = A.blk[bk], b1 = A.blk[bk + 1];
    const int r0 = b0.x, nr = b1.x - b0.x;
    const int ea = b0.y & ~3;              // 4-entry aligned start: 16 B (col) / 32 B (val) aligned
    const int n4 = (b1.y - ea + 3) >> 2;   // 4-entry groups to stream (<= S_STEPS * BLOCK by construction)
    // prefetch row extents and the first chunk's epilogue operands; their latency overlaps phase A
    int pb = 0, pe = 0;
    unsigned char sk = 0;
    double e_in0 = 0.0, e_in1 = 0.0, e_w = 0.0, e_aux = 0.0, e_dot = 0.0;
    if (t < nr) {
      const int row = r0 + t;
      pb = A.ptr[row] - ea;
      pe = A.ptr[row + 1] - ea;
      if (fh.skip) sk = fh.skip[row];
      if (MODE == M_RESID || MODE == M_JACOBI || MODE == M_ADD || MODE == M_CHEB) e_in0 = a.in0[row];
      if (MODE == M_JACOBI || MODE == M_CHEB) e_in1 = a.in1[row];
      if (MODE == M_JACOBI || MODE == M_CHEB || (MODE == M_RESTRICT && a.out2)) e_w = a.w[row];
      if (MODE == M_CHEB && a.aux) e_aux = a.aux[row];
      if (DOT) e_dot = a.dotv[row];
    }
    // phase A: stream entries [ea, ea + 4 n4).  Entries outside the block's own range belong to the
    // neighbouring blocks (or the zero padding): valid data, their products are simply never read.
    const int4* __restrict__ col4 = reinterpret_cast<const int4*>(A.col + ea);
    const double2* __restrict__ val2 = reinterpret_cast<const double2*>(A.val + ea);
    int4 c[S_STEPS];
    double2 v0[S_STEPS], v1[S_STEPS];
#pragma unroll
    for (int j = 0; j < S_STEPS; ++j) {
      const int g = t + j * BLOCK;
      if (g < n4) {
        c[j] = __ldcs(col4 + g);
        v0[j] = __ldcs(val2 + 2 * g);
        v1[j] = __ldcs(val2 + 2 * g + 1);
      }
    }
#pragma unroll
    for (int j = 0; j < S_STEPS; ++j) {
      const int g = t + j * BLOCK;
      if (g < n4) {
        const double x0 = x[c[j].x], x1 = x[c[j].y], x2 = x[c[j].z], x3 = x[c[j].w];
        double2 p0, p1;
        p0.x = v0[j].x * x0;
        p0.y = v0[j].y * x1;
        p1.x = v1[j].x * x2;
        p1.y = v1[j].y * x3;
        reinterpret_cast<double2*>(prod)[2 * g] = p0;
        reinterpret_cast<double2*>(prod)[2 * g + 1] = p1;
      }
    }
    __syncthreads();
    if (LONG) {  // S_LB lanes per row, BLOCK / S_LB rows per pass (block-uniform trip count: full-mask shuffles)
      constexpr int S_LB = 16;
      const int lane = t & (S_LB - 1);
      for (int rr0 = 0; rr0 < nr; rr0 += BLOCK / S_LB) {
        const int rr = rr0 + t / S_LB;
        const bool valid = rr < nr;
        const int row = r0 + rr;
        int qb = 0, qe = 0;
        unsigned char sk2 = 0;
        double f_in0 = 0.0, f_in1 = 0.0, f_w = 0.0, f_aux = 0.0, f_dot = 0.0;
        if (valid) {
          qb = A.ptr[row] - ea;
          qe = A.ptr[row + 1] - ea;
          if (lane == 0) {  // the epilogue operands travel while the lanes add
            if (fh.skip) sk2 = fh.skip[row];
            if (MODE == M_RESID || MODE == M_JACOBI || MODE == M_ADD || MODE == M_CHEB) f_in0 = a.in0[row];
            if (MODE == M_JACOBI || MODE == M_CHEB) f_in1 = a.in1[row];
            if (MODE == M_JACOBI || MODE == M_CHEB || (MODE == M_RESTRICT && a.out2)) f_w = a.w[row];
            if (MODE == M_CHEB && a.aux) f_aux = a.aux[row];
            if (DOT) f_dot = a.dotv[row];
          }
        }
        double s = 0.0;
        for (int k = qb + lane; k < qe; k += S_LB) s += prod[k];
#pragma unroll
        for (int o = S_LB / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (valid && lane == 0 && !sk2) {
          const double res = stream_epilogue<MODE>(a, row, s, f_in0, f_in1, f_w, f_aux);
          if (DOT) acc += f_dot * res;
        }
      }
    } else
    // phase B: thread t owns rows t, t + BLOCK, ...; products summed in column order
#pragma unroll
    for (int q = 0; q < S_CHUNKS; ++q) {
      const int rr = t + q * BLOCK;
      if (rr < nr) {
        const int row = r0 + rr;
        if (q > 0) {  // extents / operands of the later chunks (short-row matrices only) are fetched here
          pb = A.ptr[row] - ea;
          pe = A.ptr[row + 1] - ea;
          if (fh.skip) sk = fh.skip[row];
          if (MODE == M_RESID || MODE == M_JACOBI || MODE == M_ADD || MODE == M_CHEB) e_in0 = a.in0[row];
          if (MODE == M_JACOBI || MODE == M_CHEB) e_in1 = a.in1[row];
          if (MODE == M_JACOBI || MODE == M_CHEB || (MODE == M_RESTRICT && a.out2)) e_w = a.w[row];
          if (MODE == M_CHEB && a.aux) e_aux = a.aux[row];
          if (DOT) e_dot = a.dotv[row];
        }
        double s = 0.0;
        for (int k = pb; k < pe; ++k) s += prod[k];
        if (!sk) {
          const double res = stream_epilogue<MODE>(a, row, s, e_in0, e_in1, e_w, e_aux);
          if (DOT) acc += e_dot * res;
        }
      }
    }
    if (bk + n_main < A.nblocks) __syncthreads();  // prod is reused by the next row block
  }
  if (DOT) dot_finish(acc, partials, st, &st->ticket[0], rc, publish, 0, red_slot);
}

// ---------------------------------------------------------------------------------------------
// SELL-C-sigma SpMV family.  C = 32 * RPT rows per slice = one warp; lane l owns RPT adjacent rows
// of the slice.  Slice storage is column-major: entry j of the slice's rows is one contiguous,
// aligned run of C values (and C column ids), so a warp's load of entry j is one fully coalesced
// 256 B * RPT (values) / 128 B * RPT (column ids) transaction -- 128-bit per thread for the values
// when RPT = 2 -- and there is no row pointer, no shared memory and no cross-lane reduction.
// Rows are sorted by length (descending, stable) inside windows of sigma rows before slicing, which
// bounds the padding for the variable-length rows of P and R; `perm` maps a slot back to its row.
// Padding entries are (value 0.0, column = a valid column of the row): they add +0.0.
// A row is summed sequentially in column order with the product rounded before the addition
// (__dmul_rn / __dadd_rn: no FMA contraction), i.e. bit-identically to the oracle's CSR loop.
// ---------------------------------------------------------------------------------------------
struct SellView {
  const int32_t* slice_off;  // [nslices + 1] first entry-row of each slice, in units of C entries
  const int32_t* col;        // [slice_off[nslices] * C]
  const double* val;
  const int32_t* perm;       // slot -> row, or nullptr (identity)
  int32_t nrows, nslices;
};

template <int RPT>
struct SellVec;
template <>
struct SellVec<1> {
  using V = double;
  using I = int32_t;
};
template <>
struct SellVec<2> {
  using V = double2;
  using I = int2;
};
__device__ __forceinline__ double sv_get(const double& v, int) { return v; }
__device__ __forceinline__ double sv_get(const double2& v, int k) { return k ? v.y : v.x; }
__device__ __forceinline__ int sv_get(const int32_t& v, int) { return v; }
__device__ __forceinline__ int sv_get(const int2& v, int k) { return k ? v.y : v.x; }

// U: entries of a row in flight per step; MINB: resident CTAs per SM the register budget must allow (RPT = 2: 4 x 128-bit value
// loads + 4 x 64-bit column loads per thread and step, 3 CTAs/SM).
template <int RPT, int MODE, bool DOT, int U = (RPT == 1 ? 8 : 4), int MINB = (RPT == 1 ? 4 : 3)>
__global__ void __launch_bounds__(BLOCK, MINB) k_spmv_sell(SellView A, const double* __restrict__ x, EpiArgs a, DevState* st,
                                                      FusedHalo fh, double* partials, RedCtx rc, int publish, int red_slot) {
  if (st->done) return;
  trace_mark(st);
  const int n_main = (int)gridDim.x - fh.n_pack - fh.n_bnd;
  const int bid = (int)blockIdx.x - fh.n_pack - (fh.bnd_first ? fh.n_bnd : 0);
  const int b0 = fh.n_pack + (fh.bnd_first ? 0 : n_main);  // first boundary CTA
  if ((int)blockIdx.x < fh.n_pack || ((int)blockIdx.x >= b0 && (int)blockIdx.x < b0 + fh.n_bnd)) {  // halo roles
    double racc = 0.0;
    if ((int)blockIdx.x < fh.n_pack)
      pack_role(fh, st, blockIdx.x);
    else
      racc = boundary_role<MODE, DOT>(fh, x, a, st, (int)blockIdx.x - b0);
    if (DOT) dot_finish(racc, partials, st, &st->ticket[0], rc, publish, 0, red_slot);
    return;
  }
  using V = typename SellVec<RPT>::V;
  using I = typename SellVec<RPT>::I;
  const int lane = threadIdx.x & 31;
  const int wpb = BLOCK / 32;
  __shared__ double s_acc[DOT ? BLOCK : 1];  // per-thread running dot (each thread touches only its own slot)
  if (DOT) s_acc[threadIdx.x] = 0.0;
  for (int sl = bid * wpb + (threadIdx.x >> 5); sl < A.nslices; sl += n_main * wpb) {
    const int o0 = A.slice_off[sl], w = A.slice_off[sl + 1] - o0;
    const int slot0 = sl * (32 * RPT) + lane * RPT;
    // Nothing but the row sums stays in registers across the entry loop: the epilogue operands, the skip
    // flags and (with a permutation) the row ids are prefetched into L1 here and loaded after the loop.
#pragma unroll
    for (int k = 0; k < RPT; ++k) {
      const int slot = slot0 + k;
      if (slot < A.nrows) {
        const int r = A.perm ? A.perm[slot] : slot;
        if (fh.skip) asm volatile("prefetch.global.L1 [%0];" ::"l"(fh.skip + r));
        if (MODE == M_RESID || MODE == M_JACOBI || MODE == M_ADD || MODE == M_CHEB) prefetch_l1(a.in0 + r);
        if (MODE == M_JACOBI || MODE == M_CHEB || (MODE == M_RESTRICT && a.out2)) prefetch_l1(a.w + r);
        if (MODE == M_CHEB && a.aux) prefetch_l1(a.aux + r);
        if (DOT && a.dotv != a.in0) prefetch_l1(a.dotv + r);
      }
    }
    double s[RPT];
#pragma unroll
    for (int k = 0; k < RPT; ++k) s[k] = 0.0;
    const V* __restrict__ vj = reinterpret_cast<const V*>(A.val) + (size_t)o0 * 32 + lane;
    const I* __restrict__ cj = reinterpret_cast<const I*>(A.col) + (size_t)o0 * 32 + lane;
#pragma unroll 1
    for (int j0 = 0; j0 < w; j0 += U, vj += U * 32, cj += U * 32) {
      V v[U];
      I c[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
          c[u] = __ldcs(cj + u * 32);
          v[u] = __ldcs(vj + u * 32);
        }
      double xv[U][RPT];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
#pragma unroll
          for (int k = 0; k < RPT; ++k) xv[u][k] = x[sv_get(c[u], k)];
        }
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
#pragma unroll
          for (int k = 0; k < RPT; ++k) s[k] = __dadd_rn(s[k], __dmul_rn(sv_get(v[u], k), xv[u][k]));
        }
    }
    double contrib = 0.0;
#pragma unroll
    for (int k = 0; k < RPT; ++k) {
      const int slot = slot0 + k;
      if (slot < A.nrows) {
        const int r = A.perm ? A.perm[slot] : slot;
        if (fh.skip && fh.skip[r]) continue;
        const double res = apply_epilogue<MODE, false>(a, r, s[k]);
        if (DOT) contrib += a.dotv[r] * res;  // after the stores: an L1 hit (prefetched above), and it keeps ptxas batching the loop loads
      }
    }
    if (DOT) s_acc[threadIdx.x] += contrib;  // in shared memory: a register live across the entry loop costs its load batching
  }
  if (DOT) dot_finish(s_acc[threadIdx.x], partials, st, &st->ticket[0], rc, publish, 0, red_slot);
}

// ---------------------------------------------------------------------------------------------
// Value-indexed SELL (RPT = 2).  An operator with at most 256 DISTINCT values -- the 7-point Poisson matrix has two, its
// smoothed-aggregation prolongator and restriction nine -- is stored as int32 columns + one byte per entry that indexes a
// dictionary of the distinct fp64 values (CSR-VI, Kourtis et al.): 5 bytes per entry instead of 12 cross the HBM pins.  The
// dictionary (<= 2 KB) sits in shared memory; every product is __dmul_rn(dict[i], x[c]) with the ORIGINAL double, summed in
// the same order, so results are bit-identical to the fp64-valued kernel.  Layout of the indices = layout of the columns
// (entry j of slot q at (slice_off[sl] + j) * 64 + q): a lane reads its two rows' indices with one 16-bit load.
// A kernel of its own so that the fp64-valued production instantiations keep their registers and load schedule.  Blocks whose
// rows were sorted (permuted) run this two-rows-per-lane kernel; unsorted ones run k_spmv_sell_vi4 below.
// ---------------------------------------------------------------------------------------------
struct SellViView {
  const int32_t* slice_off;
  const int32_t* col;
  const uint8_t* vidx;   // [slice_off[nslices] * C] dictionary index per stored entry (padding -> the entry holding 0.0); one byte each,
                         // two (little endian) in the wide form of k_spmv_sell_vi4
  const double* dict;    // [256], wide form: [ndict]
  const int32_t* perm;
  int32_t nrows, nslices;
  int32_t ndict;         // dictionary entries (wide form: <= VI_WIDE_MAX, copied to dynamic shared memory)
};
constexpr int VI_WIDE_MAX = 4096;  // 32 KB of shared memory per CTA

// 4 entries of a row in flight per step, 3 CTAs/SM
template <int MODE, bool DOT>
__global__ void __launch_bounds__(BLOCK, 3) k_spmv_sell_vi(SellViView A, const double* __restrict__ x, EpiArgs a, DevState* st, FusedHalo fh,
                                                         double* partials, RedCtx rc, int publish, int red_slot) {
  constexpr int U = 4;
  if (st->done) return;
  trace_mark(st);
  const int n_main = (int)gridDim.x - fh.n_pack - fh.n_bnd;
  const int bid = (int)blockIdx.x - fh.n_pack - (fh.bnd_first ? fh.n_bnd : 0);
  const int b0 = fh.n_pack + (fh.bnd_first ? 0 : n_main);  // first boundary CTA
  if ((int)blockIdx.x < fh.n_pack || ((int)blockIdx.x >= b0 && (int)blockIdx.x < b0 + fh.n_bnd)) {  // halo roles
    double racc = 0.0;
    if ((int)blockIdx.x < fh.n_pack)
      pack_role(fh, st, blockIdx.x);
    else
      racc = boundary_role<MODE, DOT>(fh, x, a, st, (int)blockIdx.x - b0);
    if (DOT) dot_finish(racc, partials, st, &st->ticket[0], rc, publish, 0, red_slot);
    return;
  }
  __shared__ double s_dict[256];
  __shared__ double s_acc[DOT ? BLOCK : 1];
  s_dict[threadIdx.x] = A.dict[threadIdx.x];  // BLOCK == 256
  if (DOT) s_acc[threadIdx.x] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wpb = BLOCK / 32;
  for (int sl = bid * wpb + (threadIdx.x >> 5); sl < A.nslices; sl += n_main * wpb) {
    const int o0 = A.slice_off[sl], w = A.slice_off[sl + 1] - o0;
    const int slot0 = sl * 64 + lane * 2;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int slot = slot0 + k;
      if (slot < A.nrows) {
        const int r = A.perm ? A.perm[slot] : slot;
        if (fh.skip) asm volatile("prefetch.global.L1 [%0];" ::"l"(fh.skip + r));
        if (MODE == M_RESID || MODE == M_JACOBI || MODE == M_ADD || MODE == M_CHEB) prefetch_l1(a.in0 + r);
        if (MODE == M_JACOBI || MODE == M_CHEB || (MODE == M_RESTRICT && a.out2)) prefetch_l1(a.w + r);
        if (MODE == M_CHEB && a.aux) prefetch_l1(a.aux + r);
        if (DOT && a.dotv != a.in0) prefetch_l1(a.dotv + r);
      }
    }
    double s0 = 0.0, s1 = 0.0;
    const int2* __restrict__ cj = reinterpret_cast<const int2*>(A.col) + (size_t)o0 * 32 + lane;
    const unsigned short* __restrict__ ij = reinterpret_cast<const unsigned short*>(A.vidx) + (size_t)o0 * 32 + lane;
#pragma unroll 1
    for (int j0 = 0; j0 < w; j0 += U, cj += U * 32, ij += U * 32) {
      int2 c[U];
      unsigned short iv[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
          c[u] = __ldcs(cj + u * 32);
          iv[u] = __ldcs(ij + u * 32);
        }
      double xv[U][2];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
          xv[u][0] = x[c[u].x];
          xv[u][1] = x[c[u].y];
        }
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
          s0 = __dadd_rn(s0, __dmul_rn(s_dict[iv[u] & 0xffu], xv[u][0]));
          s1 = __dadd_rn(s1, __dmul_rn(s_dict[iv[u] >> 8], xv[u][1]));
        }
    }
    double contrib = 0.0;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int slot = slot0 + k;
      if (slot < A.nrows) {
        const int r = A.perm ? A.perm[slot] : slot;
        if (fh.skip && fh.skip[r]) continue;
        const double res = apply_epilogue<MODE, false>(a, r, k ? s1 : s0);
        if (DOT) contrib += a.dotv[r] * res;
      }
    }
    if (DOT) s_acc[threadIdx.x] += contrib;
  }
  if (DOT) dot_finish(s_acc[threadIdx.x], partials, st, &st->ticket[0], rc, publish, 0, red_slot);
}

// Value-indexed SELL with FOUR rows per lane, interleaved (formats.hpp sell_layout interleave = 4): slices of 128 rows; lane l owns
// rows l, l + 32, l + 64, l + 96 of its slice.  ncu on the two-row form (256^3 SpMV, 0.21 ms for 0.83 GB): DRAM 48 %, L1 49 %,
// 6 warps per scheduler of which 0.37 eligible, 14.7 long-scoreboard stalls per issue -- latency bound with too little in
// flight.  Here a warp carries twice the rows through the same number of dependent phases (one 128-bit column load and one
// 32-bit index load per entry and lane), and because the lanes of a warp now touch 32 CONSECUTIVE rows per access the x
// gathers and the epilogue cost half the L1 wavefronts per row.  Same products, same order, same bits.
// index of row k (0..3) of a lane in the loaded index word(s); vi_bits: any function of ALL their bits (load-order dependence)
__device__ __forceinline__ unsigned vi_index(unsigned v, int k) { return (v >> (8 * k)) & 0xffu; }
__device__ __forceinline__ unsigned vi_index(const uint2& v, int k) { return ((k < 2 ? v.x : v.y) >> (16 * (k & 1))) & 0xffffu; }
__device__ __forceinline__ unsigned vi_bits(unsigned v) { return v; }
__device__ __forceinline__ unsigned vi_bits(const uint2& v) { return v.x | v.y; }

// The four rows of a lane in the 128-row layouts: r_first + k rstep, k = 0..3 (rstep 32 in a full slice, 1 in the partial last one).
// Their epilogue operands are requested into L1 before the entry loop ...
template <int MODE, bool DOT>
__device__ __forceinline__ void rows4_prefetch(const EpiArgs& a, const FusedHalo& fh, int r_first, int rstep, int nrows) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int r = r_first + k * rstep;
    if (r < nrows) {
      if (fh.skip) asm volatile("prefetch.global.L1 [%0];" ::"l"(fh.skip + r));
      if (MODE == M_RESID || MODE == M_JACOBI || MODE == M_ADD || MODE == M_CHEB) prefetch_l1(a.in0 + r);
      if (MODE == M_JACOBI || MODE == M_CHEB || (MODE == M_RESTRICT && a.out2)) prefetch_l1(a.w + r);
      if (MODE == M_CHEB && a.aux) prefetch_l1(a.aux + r);
      if (DOT && a.dotv != a.in0) prefetch_l1(a.dotv + r);
    }
  }
}

// ... and the epilogue runs two rows at a time: their operand loads first (L1 hits), then arithmetic and stores.  Returns the lane's dot
// contribution, added over its rows in order k = 0..3.
template <int MODE, bool DOT>
__device__ __forceinline__ double rows4_epilogue(const EpiArgs& a, const FusedHalo& fh, const double (&s)[4], int r_first, int rstep,
                                                 int nrows) {
  double contrib = 0.0;
#pragma unroll
  for (int h = 0; h < 4; h += 2) {
    bool live[2];
    double e_in0[2], e_in1[2], e_w[2], e_aux[2], e_dot[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int r = r_first + (h + k) * rstep;
      live[k] = r < nrows && !(fh.skip && fh.skip[r]);
      e_in0[k] = e_in1[k] = e_w[k] = e_aux[k] = e_dot[k] = 0.0;
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int r = r_first + (h + k) * rstep;
      if (live[k]) {
        if (MODE == M_RESID || MODE == M_JACOBI || MODE == M_ADD || MODE == M_CHEB) e_in0[k] = a.in0[r];
        if (MODE == M_JACOBI || MODE == M_CHEB) e_in1[k] = a.in1[r];
        if (MODE == M_JACOBI || MODE == M_CHEB || (MODE == M_RESTRICT && a.out2)) e_w[k] = a.w[r];
        if (MODE == M_CHEB && a.aux) e_aux[k] = a.aux[r];
        if (DOT) e_dot[k] = (a.dotv == a.in0 && (MODE == M_JACOBI || MODE == M_RESID)) ? e_in0[k] : a.dotv[r];
      }
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int r = r_first + (h + k) * rstep;
      if (live[k]) {
        const double res = stream_epilogue<MODE>(a, r, s[h + k], e_in0[k], e_in1[k], e_w[k], e_aux[k]);
        if (DOT) contrib += e_dot[k] * res;
      }
    }
  }
  return contrib;
}

// AHEAD = 1: the extents of a warp's NEXT slice are loaded one iteration early and that slice's columns / indices are requested into L2
// (prefetch.global.L2: no register, no scoreboard), which takes the extents latency off the per-slice chain and turns the column latency
// from HBM into L2.  The engine launches four instantiations, IB x bounded: a launch capped at one resident wave of persistent CTAs runs
// AHEAD = 1, and its one-byte form U = 2 at 4 CTAs/SM (64 registers, no spill); the others run U = 4 at 3 CTAs/SM.
template <int MODE, bool DOT, int IB = 1, int U = 4, int MINB = 3, int AHEAD = 0>
__global__ void __launch_bounds__(BLOCK, MINB) k_spmv_sell_vi4(SellViView A, const double* __restrict__ x, EpiArgs a, DevState* st, FusedHalo fh,
                                                            double* partials, RedCtx rc, int publish, int red_slot) {
  if (st->done) return;
  trace_mark(st);
  const int n_main = (int)gridDim.x - fh.n_pack - fh.n_bnd;
  const int bid = (int)blockIdx.x - fh.n_pack - (fh.bnd_first ? fh.n_bnd : 0);
  const int b0 = fh.n_pack + (fh.bnd_first ? 0 : n_main);  // first boundary CTA
  if ((int)blockIdx.x < fh.n_pack || ((int)blockIdx.x >= b0 && (int)blockIdx.x < b0 + fh.n_bnd)) {  // halo roles
    double racc = 0.0;
    if ((int)blockIdx.x < fh.n_pack)
      pack_role(fh, st, blockIdx.x);
    else
      racc = boundary_role<MODE, DOT>(fh, x, a, st, (int)blockIdx.x - b0);
    if (DOT) dot_finish(racc, partials, st, &st->ticket[0], rc, publish, 0, red_slot);
    return;
  }
  // IB = 1: one index byte per entry, 256 dictionary entries; IB = 2 (wide): two bytes, up to VI_WIDE_MAX entries (the Galerkin
  // matrix of level 1 of the Poisson hierarchy has a few hundred to a few thousand distinct values: 6 instead of 12 bytes per entry)
  extern __shared__ double s_dict[];
  __shared__ double s_acc[DOT ? BLOCK : 1];
  for (int i = threadIdx.x; i < A.ndict; i += BLOCK) s_dict[i] = A.dict[i];
  if (DOT) s_acc[threadIdx.x] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wpb = BLOCK / 32;
  const int stride = n_main * wpb;
  int sl = bid * wpb + (threadIdx.x >> 5);
  int o0c = 0, wc = 0;  // AHEAD: extents of the current slice, loaded during the previous iteration
  if (AHEAD && sl < A.nslices) {
    o0c = A.slice_off[sl];
    wc = A.slice_off[sl + 1] - o0c;
  }
  for (; sl < A.nslices; sl += stride) {
    int o0, w;
    if (AHEAD) {
      o0 = o0c;
      w = wc;
      if (sl + stride < A.nslices) {
        o0c = A.slice_off[sl + stride];
        wc = A.slice_off[sl + stride + 1] - o0c;
      } else {
        wc = 0;
      }
    } else {
      o0 = A.slice_off[sl];
      w = A.slice_off[sl + 1] - o0;
    }
    const int base = sl * 128;
    const bool full = base + 128 <= A.nrows;
    // row of (lane, k): 32 apart in a full slice, adjacent in the partial last one
    const int rstep = full ? 32 : 1;
    const int r_first = full ? base + lane : base + lane * 4;
    rows4_prefetch<MODE, DOT>(a, fh, r_first, rstep, A.nrows);
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    const int4* __restrict__ cj = reinterpret_cast<const int4*>(A.col) + (size_t)o0 * 32 + lane;
    using IV = typename std::conditional<IB == 1, unsigned, uint2>::type;
    const IV* __restrict__ ij = reinterpret_cast<const IV*>(A.vidx) + (size_t)o0 * 32 + lane;
#pragma unroll 1
    for (int j0 = 0; j0 < w; j0 += U, cj += U * 32, ij += U * 32) {
      int4 c[U];
      IV iv[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
          c[u] = __ldcs(cj + u * 32);
          iv[u] = __ldcs(ij + u * 32);
        }
      // The gathers must not drift up between the column loads: ptxas interleaved them in four of the six modes (column load,
      // its four gathers, next column load, ...: one exposed latency per entry instead of one per step), and neither a
      // compiler barrier nor a warp barrier holds non-coherent loads back.  A data dependence does: the gather base is offset by
      // the sign of the OR of all the step's columns -- zero, since columns are non-negative, but not provably so.
      int allc = 0;
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) allc |= c[u].x | c[u].y | c[u].z | c[u].w | (int)(vi_bits(iv[u]) >> 1);  // the index loads too: they go out with the columns
      const int z = allc >> 31;
      double xv[U][4];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
          xv[u][0] = x[c[u].x + z];
          xv[u][1] = x[c[u].y + z];
          xv[u][2] = x[c[u].z + z];
          xv[u][3] = x[c[u].w + z];
        }
      asm volatile("" ::: "memory");
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
#pragma unroll
          for (int k = 0; k < 4; ++k) s[k] = __dadd_rn(s[k], __dmul_rn(s_dict[vi_index(iv[u], k)], xv[u][k]));
        }
    }
    if (AHEAD && wc > 0) {  // next slice of this warp: one 128-byte line per lane and request (columns: 4 lines per entry, indices: IB)
      const char* pc = reinterpret_cast<const char*>(A.col) + (size_t)o0c * 512;
      const char* pi = reinterpret_cast<const char*>(A.vidx) + (size_t)o0c * (128 * IB);
      for (int q = lane; q < wc * 4; q += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(pc + (size_t)q * 128));
      for (int q = lane; q < wc * IB; q += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(pi + (size_t)q * 128));
    }
    const double contrib = rows4_epilogue<MODE, DOT>(a, fh, s, r_first, rstep, A.nrows);
    if (DOT) s_acc[threadIdx.x] += contrib;
  }
  if (DOT) dot_finish(s_acc[threadIdx.x], partials, st, &st->ticket[0], rc, publish, 0, red_slot);
}

// SELL with implied columns (formats.hpp diag_layout): stencil operators, whose rows hold their entries at row + off[j] for at most
// SELL_DIAG_MAX fixed offsets.  A slot stores only its index byte (1 byte per slot instead of 5 per entry: at 256^3 the matrix is
// 0.117 instead of 0.585 GB per pass), and every x address is row + off[j], known before any load: no column -> gather chain, and the
// 32 lanes of a warp read 32 consecutive doubles per diagonal.  Same slice -> warp -> lane map, same per-row product order
// (ascending offset = ascending column = stored order) and the same epilogue as k_spmv_sell_vi4, so with the same grid every row result
// AND the fused dot products are bit-identical to it.  An absent slot leaves the sum untouched (the vi4 kernel's row padding adds
// +0.0 * x, which cannot change a sum that starts at +0.0 when x is finite).
constexpr int SELL_DIAG_MAX = 32;
constexpr unsigned SELL_DIAG_ABSENT = 255u;
struct SellDiagView {
  const uint32_t* idx;  // [nslices * ndiag * 32] words: byte k of word (sl * ndiag + j) * 32 + lane = row k of the lane on diagonal j
  const double* dict;   // [256]
  const int32_t* off;   // [ndiag] ascending column offsets
  int32_t nrows, nslices, ndiag;
};

// U = 2 diagonals per step: no spills at 64 registers (4 CTAs/SM, the vi4 launch's occupancy); U = 3 spills in JACOBI + DOT, U = 4 in
// five of the eight instantiations.
template <int MODE, bool DOT, int U = 2, int MINB = 4>
__global__ void __launch_bounds__(BLOCK, MINB) k_spmv_sell_diag(SellDiagView A, const double* __restrict__ x, EpiArgs a, DevState* st,
                                                              FusedHalo fh, double* partials, RedCtx rc, int publish, int red_slot) {
  if (st->done) return;
  trace_mark(st);
  const int n_main = (int)gridDim.x - fh.n_pack - fh.n_bnd;
  const int bid = (int)blockIdx.x - fh.n_pack - (fh.bnd_first ? fh.n_bnd : 0);
  const int b0 = fh.n_pack + (fh.bnd_first ? 0 : n_main);  // first boundary CTA
  if ((int)blockIdx.x < fh.n_pack || ((int)blockIdx.x >= b0 && (int)blockIdx.x < b0 + fh.n_bnd)) {  // halo roles
    double racc = 0.0;
    if ((int)blockIdx.x < fh.n_pack)
      pack_role(fh, st, blockIdx.x);
    else
      racc = boundary_role<MODE, DOT>(fh, x, a, st, (int)blockIdx.x - b0);
    if (DOT) dot_finish(racc, partials, st, &st->ticket[0], rc, publish, 0, red_slot);
    return;
  }
  __shared__ double s_dict[256];
  __shared__ int s_off[SELL_DIAG_MAX];
  __shared__ double s_acc[DOT ? BLOCK : 1];
  s_dict[threadIdx.x] = A.dict[threadIdx.x];  // BLOCK == 256
  if (threadIdx.x < A.ndiag) s_off[threadIdx.x] = A.off[threadIdx.x];
  if (DOT) s_acc[threadIdx.x] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wpb = BLOCK / 32;
  const int last = A.nrows - 1;
  for (int sl = bid * wpb + (threadIdx.x >> 5); sl < A.nslices; sl += n_main * wpb) {
    const int base = sl * 128;
    const bool full = base + 128 <= A.nrows;
    const int rstep = full ? 32 : 1;
    const int r_first = full ? base + lane : base + lane * 4;
    rows4_prefetch<MODE, DOT>(a, fh, r_first, rstep, A.nrows);
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    const uint32_t* __restrict__ ij = A.idx + (size_t)sl * A.ndiag * 32 + lane;
#pragma unroll 1
    for (int j0 = 0; j0 < A.ndiag; j0 += U) {
      unsigned iv[U];
      double xv[U][4];
      // x addresses come from the row and the offset only (clamped into the vector; an absent slot's value is never used)
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < A.ndiag) {
          iv[u] = __ldcs(ij + (j0 + u) * 32);
          const int o = s_off[j0 + u];
#pragma unroll
          for (int k = 0; k < 4; ++k) xv[u][k] = x[min(max(r_first + k * rstep + o, 0), last)];
        }
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < A.ndiag) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const unsigned v = vi_index(iv[u], k);
            if (v != SELL_DIAG_ABSENT) s[k] = __dadd_rn(s[k], __dmul_rn(s_dict[v], xv[u][k]));
          }
        }
    }
    const double contrib = rows4_epilogue<MODE, DOT>(a, fh, s, r_first, rstep, A.nrows);
    if (DOT) s_acc[threadIdx.x] += contrib;
  }
  if (DOT) dot_finish(s_acc[threadIdx.x], partials, st, &st->ticket[0], rc, publish, 0, red_slot);
}

// ---------------------------------------------------------------------------------------------
// k-wide forms of k_spmv_sell_diag and k_spmv_sell_vi4: K right-hand sides per launch (pamg_*_multi)
// ---------------------------------------------------------------------------------------------
// Per step a lane loads the index word (and for vi4 the column word) once, then gathers and accumulates for every live column.  Per
// column everything is the single kernel's: the slice -> warp -> lane map and slice stride (the engine launches the same grid), the
// per-row __dmul_rn / __dadd_rn order, rows4_prefetch / rows4_epilogue, one s_acc slot per thread, and dot_finish on the column's own
// partials, ticket and RedCtx.  So column c of a k-wide launch is bit-identical to the single kernel on column c alone.  Main role only:
// multi-column calls run their halo exchange as separate k_halo_pack / k_boundary launches per column.  A column is live when its
// pointer is set and its DevState is not `done` (a converged column is frozen as in the single-column solve).
template <int K>
struct MultiCols {
  const double* x[K];
  EpiArgs a[K];
  DevState* st[K];  // nullptr: absent column
  double* partials[K];
  RedCtx rc[K];
};

template <int K>
__device__ __forceinline__ unsigned live_columns(const MultiCols<K>& m) {
  unsigned live = 0;
#pragma unroll
  for (int c = 0; c < K; ++c)
    if (m.st[c] && !m.st[c]->done) live |= 1u << c;
  return live;
}

template <int MODE, bool DOT, int K>
__device__ __forceinline__ void multi_finish(const MultiCols<K>& m, unsigned live, double (&s_acc)[K][BLOCK], int publish, int red_slot) {
#pragma unroll
  for (int c = 0; c < K; ++c)
    if (live >> c & 1u) dot_finish(s_acc[c][threadIdx.x], m.partials[c], m.st[c], &m.st[c]->ticket[0], m.rc[c], publish, 0, red_slot);
}

// U = 1 diagonal per step at K = 4, 2 at K = 2 (scripts/ptxas_table.py: no spills)
template <int MODE, bool DOT, int K, int U = (K >= 4 ? 1 : 2), int MINB = 2>
__global__ void __launch_bounds__(BLOCK, MINB) k_spmv_sell_diag_multi(SellDiagView A, MultiCols<K> m, FusedHalo fh, int publish, int red_slot) {
  const unsigned live = live_columns(m);
  if (!live) return;
#pragma unroll
  for (int c = 0; c < K; ++c)
    if (live >> c & 1u) trace_mark(m.st[c]);
  const int n_main = (int)gridDim.x;
  __shared__ double s_dict[256];
  __shared__ int s_off[SELL_DIAG_MAX];
  __shared__ double s_acc[K][DOT ? BLOCK : 1];
  s_dict[threadIdx.x] = A.dict[threadIdx.x];  // BLOCK == 256
  if (threadIdx.x < A.ndiag) s_off[threadIdx.x] = A.off[threadIdx.x];
  if (DOT)
#pragma unroll
    for (int c = 0; c < K; ++c) s_acc[c][threadIdx.x] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wpb = BLOCK / 32;
  const int last = A.nrows - 1;
  for (int sl = blockIdx.x * wpb + (threadIdx.x >> 5); sl < A.nslices; sl += n_main * wpb) {
    const int base = sl * 128;
    const bool full = base + 128 <= A.nrows;
    const int rstep = full ? 32 : 1;
    const int r_first = full ? base + lane : base + lane * 4;
#pragma unroll
    for (int c = 0; c < K; ++c)
      if (live >> c & 1u) rows4_prefetch<MODE, DOT>(m.a[c], fh, r_first, rstep, A.nrows);
    double s[K][4];
#pragma unroll
    for (int c = 0; c < K; ++c)
#pragma unroll
      for (int k = 0; k < 4; ++k) s[c][k] = 0.0;
    const uint32_t* __restrict__ ij = A.idx + (size_t)sl * A.ndiag * 32 + lane;
#pragma unroll 1
    for (int j0 = 0; j0 < A.ndiag; j0 += U) {
      unsigned iv[U];
      double xv[K][U][4];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < A.ndiag) {
          iv[u] = __ldcs(ij + (j0 + u) * 32);
          const int o = s_off[j0 + u];
#pragma unroll
          for (int c = 0; c < K; ++c)
            if (live >> c & 1u)
#pragma unroll
              for (int k = 0; k < 4; ++k) xv[c][u][k] = m.x[c][min(max(r_first + k * rstep + o, 0), last)];
        }
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < A.ndiag) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const unsigned v = vi_index(iv[u], k);
            if (v != SELL_DIAG_ABSENT) {
              const double d = s_dict[v];
#pragma unroll
              for (int c = 0; c < K; ++c)
                if (live >> c & 1u) s[c][k] = __dadd_rn(s[c][k], __dmul_rn(d, xv[c][u][k]));
            }
          }
        }
    }
#pragma unroll
    for (int c = 0; c < K; ++c)
      if (live >> c & 1u) {
        const double contrib = rows4_epilogue<MODE, DOT>(m.a[c], fh, s[c], r_first, rstep, A.nrows);
        if (DOT) s_acc[c][threadIdx.x] += contrib;
      }
  }
  if constexpr (DOT) multi_finish<MODE, DOT, K>(m, live, s_acc, publish, red_slot);
}

// IB index bytes per entry as in k_spmv_sell_vi4; U = 1 entry per step at K = 4, 2 at K = 2
template <int MODE, bool DOT, int IB, int K, int U = (K >= 4 ? 1 : 2), int MINB = 2>
__global__ void __launch_bounds__(BLOCK, MINB) k_spmv_sell_vi4_multi(SellViView A, MultiCols<K> m, FusedHalo fh, int publish, int red_slot) {
  const unsigned live = live_columns(m);
  if (!live) return;
#pragma unroll
  for (int c = 0; c < K; ++c)
    if (live >> c & 1u) trace_mark(m.st[c]);
  const int n_main = (int)gridDim.x;
  extern __shared__ double s_dict[];
  __shared__ double s_acc[K][DOT ? BLOCK : 1];
  for (int i = threadIdx.x; i < A.ndict; i += BLOCK) s_dict[i] = A.dict[i];
  if (DOT)
#pragma unroll
    for (int c = 0; c < K; ++c) s_acc[c][threadIdx.x] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wpb = BLOCK / 32;
  for (int sl = blockIdx.x * wpb + (threadIdx.x >> 5); sl < A.nslices; sl += n_main * wpb) {
    const int o0 = A.slice_off[sl];
    const int w = A.slice_off[sl + 1] - o0;
    const int base = sl * 128;
    const bool full = base + 128 <= A.nrows;
    const int rstep = full ? 32 : 1;
    const int r_first = full ? base + lane : base + lane * 4;
#pragma unroll
    for (int c = 0; c < K; ++c)
      if (live >> c & 1u) rows4_prefetch<MODE, DOT>(m.a[c], fh, r_first, rstep, A.nrows);
    double s[K][4];
#pragma unroll
    for (int c = 0; c < K; ++c)
#pragma unroll
      for (int k = 0; k < 4; ++k) s[c][k] = 0.0;
    const int4* __restrict__ cj = reinterpret_cast<const int4*>(A.col) + (size_t)o0 * 32 + lane;
    using IV = typename std::conditional<IB == 1, unsigned, uint2>::type;
    const IV* __restrict__ ij = reinterpret_cast<const IV*>(A.vidx) + (size_t)o0 * 32 + lane;
#pragma unroll 1
    for (int j0 = 0; j0 < w; j0 += U, cj += U * 32, ij += U * 32) {
      int4 cv[U];
      IV iv[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
          cv[u] = __ldcs(cj + u * 32);
          iv[u] = __ldcs(ij + u * 32);
        }
      // the data dependence of k_spmv_sell_vi4: every gather of the step goes out after all of its column and index loads
      int allc = 0;
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) allc |= cv[u].x | cv[u].y | cv[u].z | cv[u].w | (int)(vi_bits(iv[u]) >> 1);
      const int z = allc >> 31;
      double xv[K][U][4];
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
#pragma unroll
          for (int c = 0; c < K; ++c)
            if (live >> c & 1u) {
              xv[c][u][0] = m.x[c][cv[u].x + z];
              xv[c][u][1] = m.x[c][cv[u].y + z];
              xv[c][u][2] = m.x[c][cv[u].z + z];
              xv[c][u][3] = m.x[c][cv[u].w + z];
            }
        }
      asm volatile("" ::: "memory");
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (j0 + u < w) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const double d = s_dict[vi_index(iv[u], k)];
#pragma unroll
            for (int c = 0; c < K; ++c)
              if (live >> c & 1u) s[c][k] = __dadd_rn(s[c][k], __dmul_rn(d, xv[c][u][k]));
          }
        }
    }
#pragma unroll
    for (int c = 0; c < K; ++c)
      if (live >> c & 1u) {
        const double contrib = rows4_epilogue<MODE, DOT>(m.a[c], fh, s[c], r_first, rstep, A.nrows);
        if (DOT) s_acc[c][threadIdx.x] += contrib;
      }
  }
  if constexpr (DOT) multi_finish<MODE, DOT, K>(m, live, s_acc, publish, red_slot);
}

// ---------------------------------------------------------------------------------------------
// halo pack: owner -> ghost (consistent!).  Stores into the neighbours' staging, then flags.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BLOCK) k_halo_pack(const double* __restrict__ v, const int32_t* __restrict__ send_idx,
                                                      int n_send, const SendNbr* __restrict__ nbrs, int n_nbrs,
                                                      DevState* st, int level) {
  if (st->done) return;
  trace_mark(st);
  const uint32_t e = *(volatile uint32_t*)&st->halo_epoch[level] + 1u;
  const int par = (int)(e & 1u);
  for (int k = blockIdx.x * BLOCK + threadIdx.x; k < n_send; k += gridDim.x * BLOCK) {
    int nb = 0;
    while (nb + 1 < n_nbrs && k >= nbrs[nb + 1].offset) ++nb;
    nbrs[nb].ghost[par][k - nbrs[nb].offset] = v[send_idx[k]];
  }
  __threadfence_system();
  if (last_block(&st->ticket[1])) {
    __threadfence_system();
    if (threadIdx.x < n_nbrs) st_release_sys(nbrs[threadIdx.x].flag, e);
    if (threadIdx.x == 0) st->halo_epoch[level] = e;
  }
}

// copy ghost staging of the current epoch into a caller-visible buffer (pamg_consistent)
__global__ void __launch_bounds__(BLOCK) k_halo_unpack(double* __restrict__ dst, HaloRecv hr, int n_ghost, DevState* st,
                                                        int level) {
  __shared__ int s_par;
  if (threadIdx.x == 0) s_par = halo_wait(hr, *(volatile uint32_t*)&st->halo_epoch[level], st);
  __syncthreads();
  const double* g = hr.ghost[s_par];
  for (int k = blockIdx.x * BLOCK + threadIdx.x; k < n_ghost; k += gridDim.x * BLOCK) dst[k] = __ldcv(g + k);
}

// assemble!: ghost -> owner.  Pack: this part's ghost values go to the owners' assemble staging.
struct AsmSendNbr {
  double* stage[2];  // owner's staging (double-buffered by epoch parity like the halo), offset to this part's segment
  uint32_t* flag;    // owner's flag for this part
  int32_t slot0, count;
};
__global__ void __launch_bounds__(BLOCK) k_asm_pack(const double* __restrict__ ghost_vals, const AsmSendNbr* __restrict__ nbrs,
                                                     int n_nbrs, DevState* st, int level) {
  const uint32_t e = *(volatile uint32_t*)&st->asm_epoch[level] + 1u;
  const int par = (int)(e & 1u);
  for (int nb = 0; nb < n_nbrs; ++nb)
    for (int k = blockIdx.x * BLOCK + threadIdx.x; k < nbrs[nb].count; k += gridDim.x * BLOCK)
      nbrs[nb].stage[par][k] = ghost_vals[nbrs[nb].slot0 + k];
  __threadfence_system();
  if (last_block(&st->ticket[2])) {
    __threadfence_system();
    if (threadIdx.x < n_nbrs) st_release_sys(nbrs[threadIdx.x].flag, e);
    if (threadIdx.x == 0) st->asm_epoch[level] = e;
  }
}
// Add: own[i] += sum of the contributions listed for i (CSR by own row: ascending neighbour part,
// ascending slot => deterministic), then the caller zeroes the ghosts.
__global__ void __launch_bounds__(BLOCK) k_asm_add(double* __restrict__ own, const int32_t* __restrict__ rows,
                                                    const int32_t* __restrict__ ptr, const int32_t* __restrict__ src,
                                                    int n_rows, const double* stage0, const double* stage1, const uint32_t* flags,
                                                    int n_flags, DevState* st, int level) {
  __shared__ int s_par;
  if (threadIdx.x == 0) {
    const uint32_t e = *(volatile uint32_t*)&st->asm_epoch[level];
    spin_until_all(flags, n_flags, e, st);
    s_par = (int)(e & 1u);
  }
  __syncthreads();
  const double* stage = s_par ? stage1 : stage0;
  for (int r = blockIdx.x * BLOCK + threadIdx.x; r < n_rows; r += gridDim.x * BLOCK) {
    double s = own[rows[r]];
    for (int k = ptr[r]; k < ptr[r + 1]; ++k) s += __ldcv(stage + src[k]);
    own[rows[r]] = s;
  }
}

// ---------------------------------------------------------------------------------------------
// coarsest level: all-gather b_L by gid into every part, then x = A_L^-1 b (own + ghost rows)
// ---------------------------------------------------------------------------------------------
struct CoarsePub {
  double* buf[2];
  uint32_t* flag;
};
__global__ void __launch_bounds__(BLOCK) k_coarse_gather(const double* __restrict__ b, const int64_t* __restrict__ own_gid,
                                                          int n_own, const CoarsePub* __restrict__ pubs, int nparts,
                                                          DevState* st) {
  if (st->done) return;
  trace_mark(st);
  const uint32_t e = *(volatile uint32_t*)&st->coarse_epoch + 1u;
  const int par = (int)(e & 1u);
  for (int d = 0; d < nparts; ++d)
    for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n_own; i += gridDim.x * BLOCK) pubs[d].buf[par][own_gid[i]] = b[i];
  __threadfence_system();
  if (last_block(&st->ticket[3])) {
    __threadfence_system();
    if (threadIdx.x < nparts) st_release_sys(pubs[threadIdx.x].flag, e);
    if (threadIdx.x == 0) st->coarse_epoch = e;
  }
}

// one warp per output row; rows = own gids then ghost gids; ghost results go to `xg`
__global__ void __launch_bounds__(BLOCK) k_coarse_solve(const double* __restrict__ inv, int n, const double* cbuf0,
                                                         const double* cbuf1, const uint32_t* flags, int nparts,
                                                         const int64_t* __restrict__ own_gid, int n_own,
                                                         const int64_t* __restrict__ ghost_gid, int n_ghost,
                                                         double* __restrict__ x, double* __restrict__ xg, DevState* st) {
  if (st->done) return;
  trace_mark(st);
  __shared__ int s_par;
  if (threadIdx.x == 0) {
    const uint32_t e = *(volatile uint32_t*)&st->coarse_epoch;
    spin_until_all(flags, nparts, e, st);
    s_par = (int)(e & 1u);
  }
  __syncthreads();
  const double* b = s_par ? cbuf1 : cbuf0;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * BLOCK + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * BLOCK) >> 5;
  for (int r = warp; r < n_own + n_ghost; r += nwarps) {
    const int64_t g = r < n_own ? own_gid[r] : ghost_gid[r - n_own];
    const double* row = inv + (size_t)g * n;
    double s = 0.0;
    for (int j = lane; j < n; j += 32) s += row[j] * __ldcv(b + j);
    s = group_sum<32>(s);
    if (lane == 0) {
      if (r < n_own)
        x[r] = s;
      else
        xg[r - n_own] = s;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// replicated coarse tail (coarse-level agglomeration): below a size threshold every GPU holds the
// whole level (all parts merged, gid numbering) and runs it alone, with no halo at all.
//   k_coarse_gather : every part stores its slice of b into every part's gather buffer (+ flag)
//   k_tail_in       : wait for all slices; b_full <- gather buffer; first zero-guess smoothing step
//   ... the ordinary SpMV-family kernels on the merged matrices, k_dense on the coarsest level ...
//   k_tail_out      : x_full -> this part's own slice and ghost staging (prolongation to the last
//                     distributed level needs no exchange)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BLOCK) k_tail_in(const double* g0, const double* g1, const uint32_t* flags, int nparts,
                                                    double* __restrict__ b, double* __restrict__ xstart,
                                                    const double* __restrict__ w, int n, DevState* st) {
  if (st->done) return;
  trace_mark(st);
  __shared__ int s_par;
  if (threadIdx.x == 0) {
    const uint32_t e = *(volatile uint32_t*)&st->coarse_epoch;
    spin_until_all(flags, nparts, e, st);
    s_par = (int)(e & 1u);
  }
  __syncthreads();
  const double* g = s_par ? g1 : g0;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) {
    const double v = __ldcv(g + i);
    b[i] = v;
    if (xstart) xstart[i] = w ? w[i] * v : 0.0;
  }
}

// x = inv * b, one warp per row (coarsest level of the replicated tail)
__global__ void __launch_bounds__(BLOCK) k_dense(const double* __restrict__ inv, int n, const double* __restrict__ b,
                                                  double* __restrict__ x, DevState* st) {
  if (st->done) return;
  trace_mark(st);
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * BLOCK + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * BLOCK) >> 5;
  for (int r = warp; r < n; r += nwarps) {
    const double* row = inv + (size_t)r * n;
    double s = 0.0;
    for (int j = lane; j < n; j += 32) s += row[j] * b[j];
    s = group_sum<32>(s);
    if (lane == 0) x[r] = s;
  }
}

__global__ void __launch_bounds__(BLOCK) k_tail_out(const double* __restrict__ xfull, const int64_t* __restrict__ own_gid, int n_own,
                                                     const int64_t* __restrict__ ghost_gid, int n_ghost, double* __restrict__ x,
                                                     double* __restrict__ xg, DevState* st) {
  if (st->done) return;
  trace_mark(st);
  for (int r = blockIdx.x * BLOCK + threadIdx.x; r < n_own + n_ghost; r += gridDim.x * BLOCK) {
    if (r < n_own)
      x[r] = xfull[own_gid[r]];
    else
      xg[r - n_own] = xfull[ghost_gid[r - n_own]];
  }
}

// ---------------------------------------------------------------------------------------------
// PCG vector kernels (SURVEY 8a rows a6/a7), scalars stay on the device
// ---------------------------------------------------------------------------------------------
// status record for the host (pinned, device-mapped ring): one thread
__device__ __forceinline__ void write_host_status(DevState* st, HostStat* hs) {
  if (!hs) return;  // the host polls this ring instead of copying DevState between the iterations' graphs
  const uint32_t seq = st->check_seq + 1u;
  st->check_seq = seq;
  HostStat* h = hs + (seq % HS_RING);
  h->done = st->done;
  h->error = st->error;
  h->iters = st->iters;
  __threadfence_system();
  *(volatile uint32_t*)&h->seq = seq;
}

// one thread: consume ||r||^2; record history; decide convergence (identically on every part)
__device__ __forceinline__ void pcg_check(DevState* st, const RedCtx& rc, double* hist) {
  double v[RED_W];
  red_consume(st, rc, v);
  const double rr = v[0];
  const int it = st->iters + 1;
  st->iters = it;
  if (it == 0) st->sc[SC_RR0] = rr;
  st->sc[SC_RR] = rr;
  if (hist) hist[it] = sqrt(rr);
  const double rtol = st->sc[SC_RTOL];  // same test as the oracle: ||r|| <= rtol ||r0||
  if (sqrt(rr) <= rtol * sqrt(st->sc[SC_RR0]) || it >= st->maxiter) st->done = 1;
}

// the same as its own launch (several parts on one GPU: a kernel must not wait for a later kernel of its stream)
__global__ void k_check(DevState* st, RedCtx rc, double* hist, HostStat* hs) {
  if (!st->done) {
    trace_mark(st);
    pcg_check(st, rc, hist);
  }
  write_host_status(st, hs);
}

// x = 0, r = b, p = 0, z0 = w .* b (or 0), rr0 partial -> publish
__global__ void __launch_bounds__(BLOCK) k_pcg_init(const double* __restrict__ b, double* __restrict__ x, double* __restrict__ r,
                                                     double* __restrict__ p, double* __restrict__ z0, const double* __restrict__ w,
                                                     int n, DevState* st, double* partials, RedCtx rc, double rtol, int maxiter,
                                                     int fold_check, double* hist, HostStat* hs) {
  trace_mark(st);
  double acc = 0.0;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) {
    const double bi = b[i];
    x[i] = 0.0;
    r[i] = bi;
    p[i] = 0.0;
    z0[i] = w ? w[i] * bi : 0.0;
    acc += bi * bi;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    st->done = 0;
    st->check_seq = 0;
    st->iters = -1;  // the first k_check (of r0) brings it to 0
    st->maxiter = maxiter;
    st->sc[SC_RHO_OLD] = __longlong_as_double(0x7ff0000000000000ll);  // +inf => first beta = 0
    st->sc[SC_RTOL] = rtol;
  }
  // (block 0 wrote the fields above before its own ticket, and the last block has seen every ticket)
  if (dot_finish(acc, partials, st, &st->ticket[0], rc, 1, 0, 0) && fold_check) {
    pcg_check(st, rc, hist);  // ||r0||: brings iters to 0; done if b == 0 or maxiter == 0
    write_host_status(st, hs);
  }
}

// beta = rz / rho_old ; p = z + beta p
// flexible: beta = (r.z - r_prev.z) / rho_old  (Polak-Ribiere form of flexible CG; slots 1 and 3 of one all-reduce)
__global__ void __launch_bounds__(BLOCK) k_update_p(const double* __restrict__ z, double* __restrict__ p, int n, DevState* st,
                                                     RedCtx rc, int flexible) {
  if (st->done) return;
  trace_mark(st);
  __shared__ double s_beta;
  if (threadIdx.x == 0) {
    double v[RED_W];
    red_consume(st, rc, v);
    s_beta = (flexible ? v[1] - v[3] : v[1]) / st->sc[SC_RHO_OLD];
    if (blockIdx.x == 0) st->sc[SC_RHO_NEW] = v[1];
  }
  __syncthreads();
  const double beta = s_beta;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) p[i] = z[i] + beta * p[i];
}

// alpha = rho / pq ; x += alpha p ; r -= alpha q ; z0 = w .* r ; rr partial -> publish
__global__ void __launch_bounds__(BLOCK) k_update_xr(double* __restrict__ x, double* __restrict__ r, const double* __restrict__ p,
                                                      const double* __restrict__ q, double* __restrict__ z0,
                                                      const double* __restrict__ w, int n, DevState* st, double* partials,
                                                      RedCtx rc, int fold_check, double* hist, HostStat* hs,
                                                      double* __restrict__ rprev) {
  // fold_check (every part alone on its GPU): the block that publishes ||r||^2 also consumes the all-reduce and takes the
  // convergence decision, instead of a k_check launch behind this kernel
  if (st->done) {
    if (fold_check && blockIdx.x == 0 && threadIdx.x == 0) write_host_status(st, hs);  // the host still sees every iteration
    return;
  }
  trace_mark(st);
  __shared__ double s_alpha;
  if (threadIdx.x == 0) {
    double v[RED_W];
    red_consume(st, rc, v);
    s_alpha = st->sc[SC_RHO_NEW] / v[2];
  }
  __syncthreads();
  const double alpha = s_alpha;
  double acc = 0.0;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) {
    x[i] += alpha * p[i];
    const double ro = r[i];
    if (rprev) rprev[i] = ro;  // flexible CG keeps r_k for beta
    const double ri = ro - alpha * q[i];
    r[i] = ri;
    z0[i] = w ? w[i] * ri : 0.0;
    acc += ri * ri;
  }
  // every block has read RHO_NEW before the last block (which has seen all tickets) rotates it
  const double bs = block_sum(acc);
  if (threadIdx.x == 0) partials[blockIdx.x] = bs;
  if (last_block(&st->ticket[0])) {
    double s = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += BLOCK) s += __ldcv(partials + i);
    s = block_sum(s);
    if (threadIdx.x == 0) {
      st->sc[SC_RHO_OLD] = st->sc[SC_RHO_NEW];
      double v[RED_W] = {s, 0.0, 0.0, 0.0};
      red_publish(st, rc, v);
      if (fold_check) {
        pcg_check(st, rc, hist);
        write_host_status(st, hs);
      }
    }
  }
}

// plain (no preconditioner) variant support: z = r
__global__ void __launch_bounds__(BLOCK) k_copy_dot(const double* __restrict__ r, double* __restrict__ z, int n, DevState* st,
                                                     double* partials, RedCtx rc) {
  if (st->done) return;
  trace_mark(st);
  double acc = 0.0;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) {
    const double ri = r[i];
    z[i] = ri;
    acc += ri * ri;
  }
  dot_finish(acc, partials, st, &st->ticket[0], rc, 1, 0, 1);
}

__global__ void __launch_bounds__(BLOCK) k_copy(const double* __restrict__ src, double* __restrict__ dst, int n, DevState* st) {
  if (st->done) return;
  trace_mark(st);
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) dst[i] = src[i];
}

// out = w .* b  (zero-guess first Jacobi sweep) or out = 0 when w == nullptr
__global__ void __launch_bounds__(BLOCK) k_scale(const double* __restrict__ b, const double* __restrict__ w, double* __restrict__ out,
                                                  int n, DevState* st) {
  if (st->done) return;
  trace_mark(st);
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) out[i] = w ? w[i] * b[i] : 0.0;
}

// standalone dot: publishes sum(u .* v) in all-reduce slot `slot` (3 = pamg_dot, 1 = r.z)
__global__ void __launch_bounds__(BLOCK) k_dot(const double* __restrict__ u, const double* __restrict__ v, int n, DevState* st,
                                                double* partials, RedCtx rc, int slot, int honor_done) {
  if (honor_done && st->done) return;
  trace_mark(st);
  double acc = 0.0;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) acc += u[i] * v[i];
  dot_finish(acc, partials, st, &st->ticket[0], rc, 1, 0, slot);
}
// flexible CG: r.z (slot 1) and r_prev.z (slot 3) in one pass and one all-reduce
__global__ void __launch_bounds__(BLOCK) k_dot2(const double* __restrict__ r, const double* __restrict__ z,
                                                 const double* __restrict__ rprev, int n, DevState* st, double* partials, RedCtx rc) {
  if (st->done) return;
  trace_mark(st);
  double a1 = 0.0, a3 = 0.0;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) {
    const double zi = z[i];
    a1 += r[i] * zi;
    a3 += rprev[i] * zi;
  }
  const double b1 = block_sum(a1);
  const double b3 = block_sum(a3);
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = b1;
    partials[gridDim.x + blockIdx.x] = b3;
  }
  if (last_block(&st->ticket[0])) {
    double s1 = 0.0, s3 = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += BLOCK) {
      s1 += __ldcv(partials + i);
      s3 += __ldcv(partials + gridDim.x + i);
    }
    s1 = block_sum(s1);
    s3 = block_sum(s3);
    if (threadIdx.x == 0) {
      double v[RED_W] = {0.0, s1, 0.0, s3};
      red_publish(st, rc, v);
    }
  }
}
// ---------------------------------------------------------------------------------------------
// FGMRES vector kernels (SURVEY 8f rank 3; oracle/amg_oracle.py fgmres).  The Arnoldi coefficients stay on the device between
// the dot that produces them and the update that consumes them (the same publish / consume pair as PCG's scalars); the host
// reads one Hessenberg column per inner step for the Givens rotations and the convergence decision.
// ---------------------------------------------------------------------------------------------
// dst = src / d
__global__ void __launch_bounds__(BLOCK) k_div(const double* src, double* dst, double d, int n, DevState* st) {
  trace_mark(st);
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) dst[i] = __ddiv_rn(src[i], d);
}
// modified Gram-Schmidt step: h = <w, v> (slot 3 of the all-reduce published by the k_dot before) ; w -= h v ; hcol[0] = h
__global__ void __launch_bounds__(BLOCK) k_gs_sub(double* __restrict__ w, const double* __restrict__ v, int n, DevState* st, RedCtx rc,
                                                   double* hcol) {
  trace_mark(st);
  __shared__ double s_h;
  if (threadIdx.x == 0) {
    double r[RED_W];
    red_consume(st, rc, r);
    s_h = r[3];
    if (blockIdx.x == 0) hcol[0] = r[3];
  }
  __syncthreads();
  const double h = s_h;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) w[i] = __dsub_rn(w[i], __dmul_rn(h, v[i]));
}
// h_{j+1,j} = sqrt(<w, w>) ; v_{j+1} = w / h_{j+1,j} (in place; left as it is when the norm is 0: a lucky breakdown)
__global__ void __launch_bounds__(BLOCK) k_gs_norm(double* __restrict__ w, int n, DevState* st, RedCtx rc, double* hcol) {
  trace_mark(st);
  __shared__ double s_h;
  if (threadIdx.x == 0) {
    double r[RED_W];
    red_consume(st, rc, r);
    s_h = sqrt(r[3]);
    if (blockIdx.x == 0) hcol[0] = s_h;
  }
  __syncthreads();
  const double h = s_h;
  if (h == 0.0) return;
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) w[i] = __ddiv_rn(w[i], h);
}
// x += a z
__global__ void __launch_bounds__(BLOCK) k_axpy(double* __restrict__ x, const double* __restrict__ z, double a, int n, DevState* st) {
  trace_mark(st);
  for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) x[i] = __dadd_rn(x[i], __dmul_rn(a, z[i]));
}

__global__ void k_red_read(DevState* st, RedCtx rc, double* out4) {
  double v[RED_W];
  red_consume(st, rc, v);
  for (int k = 0; k < RED_W; ++k) out4[k] = v[k];
}

// L2 flush helper for timing: touch a buffer larger than L2
__global__ void k_flush(double* buf, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) buf[i] += 1.0;
}

}  // namespace pamg
