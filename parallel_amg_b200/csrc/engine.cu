// engine.cu — device-resident hierarchy, halo/all-reduce wiring over peer memory, V-cycle and
// PCG schedules (CUDA graphs), behind the C ABI of include/pamg.h.
//
// Layout in HBM, per (level, part): the own-own blocks of A, P, R in SELL-C-sigma, CSR-stream or plain CSR
// (fp64 values, int32 local columns; formats.hpp), the rows that also have own-ghost entries once more as
// whole "boundary rows", smoother weights, and own-length work vectors.  Ghost values never live in the
// vectors: they arrive in a per-level, double-buffered staging area inside the part's peer-visible
// "arena", written directly by the neighbouring GPUs.  Levels below the tail threshold exist a second
// time, merged over all parts, on every GPU (replicated coarse tail).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "engine.hpp"
#include "formats.hpp"
#include "kernels.cuh"

namespace pamg {

static_assert(DIAG_MAX_OFFSETS == SELL_DIAG_MAX && DIAG_ABSENT == SELL_DIAG_ABSENT, "formats.hpp and kernels.cuh disagree on the diagonal layout");

#define CK(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess)                                                                            \
      throw CudaError(std::string(#call) + " -> " + cudaGetErrorString(e_) + " (" + __FILE__ + ":" + \
                      std::to_string(__LINE__) + ")");                                                \
  } while (0)

namespace {

template <class T>
struct DBuf {
  T* p = nullptr;
  size_t n = 0;
  DBuf() = default;
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  ~DBuf() {
    if (p) cudaFree(p);
  }
  void alloc(size_t count, bool zero = true) {
    if (p) cudaFree(p);
    p = nullptr;
    n = count;
    CK(cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)));
    if (zero) CK(cudaMemset(p, 0, std::max<size_t>(count, 1) * sizeof(T)));
  }
  void upload(const T* h, size_t count) {
    alloc(count, false);
    if (count) CK(cudaMemcpy(p, h, count * sizeof(T), cudaMemcpyHostToDevice));
  }
  void upload(const std::vector<T>& v) { upload(v.data(), v.size()); }
};

// the buffer of the column a multi-column call is working on (Engine::Impl::bind); column 0 outside such calls
template <class T>
struct DView {
  T* p = nullptr;
  size_t n = 0;
  DView& operator=(const DBuf<T>& b) {
    p = b.p;
    n = b.n;
    return *this;
  }
};

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct DevCsr {
  DBuf<int32_t> ptr, col, rows;
  DBuf<double> val;
  int32_t nrows = 0;   // logical rows (compressed list length when `listed`)
  bool listed = false;
  int64_t nnz = 0;
  int lanes = 8;
  // CSR-stream row blocks (own-own blocks only)
  DBuf<int2> blk;
  int nblocks = 0;
  bool stream = false;
  // SELL-C-sigma (own-own blocks only)
  DBuf<int32_t> sl_off, sl_col, sl_perm;
  DBuf<double> sl_val;
  int nslices = 0, sell_rpt = 0, sell_sigma = 1;  // sell_rpt != 0 <=> the SELL kernel runs this block
  bool sell_perm = false;
  double sell_fill = 1.0;  // stored entries / nnz
  // value-indexed SELL (RPT = 2 only): one byte per stored entry into a dictionary of the <= 256 distinct values
  DBuf<uint8_t> sl_vidx;
  DBuf<double> sl_dict;
  bool sell_vi = false;
  // the same with four interleaved rows per lane (slices of 128 rows, kernels.cuh k_spmv_sell_vi4): its own slice extents / columns / indices
  DBuf<int32_t> v4_off, v4_col;
  DBuf<uint8_t> v4_idx;
  int nslices4 = 0;
  bool sell_vi4 = false;
  int vi4_ib = 1;   // bytes per index of the 128-row layout: 1 (<= 255 distinct values) or 2 (wide: <= VI_WIDE_MAX - 1)
  int ndict = 256;  // dictionary entries uploaded
  // SELL with implied columns (stencil A blocks, kernels.cuh k_spmv_sell_diag): only these arrays (and sl_dict) are uploaded
  DBuf<uint32_t> dg_idx;
  DBuf<int32_t> dg_off;
  int ndiag = 0;
  bool sell_diag = false;
  SellDiagView diagview() const { return SellDiagView{dg_idx.p, sl_dict.p, dg_off.p, nrows, nslices4, ndiag}; }
  SellViView vi4view() const { return SellViView{v4_off.p, v4_col.p, v4_idx.p, sl_dict.p, nullptr, nrows, nslices4, ndict}; }
  SellViView viview() const { return SellViView{sl_off.p, sl_col.p, sl_vidx.p, sl_dict.p, sell_perm ? sl_perm.p : nullptr, nrows, nslices, 256}; }
  CsrView view() const { return CsrView{ptr.p, col.p, val.p, listed ? rows.p : nullptr, nrows}; }
  StreamView sview() const { return StreamView{blk.p, ptr.p, col.p, val.p, nrows, nblocks}; }
  SellView slview() const { return SellView{sl_off.p, sl_col.p, sl_val.p, sell_perm ? sl_perm.p : nullptr, nrows, nslices}; }
};

// boundary rows of one operator (rows of the own-own block that also have own-ghost entries), stored
// whole for the boundary role: own-column entries then ghost-column entries
struct DevBnd {
  DBuf<int32_t> rows, ptr, mid, col;
  DBuf<double> val;
  DBuf<uint8_t> skip;  // [rows of the block] 1 = boundary row
  int n = 0, lanes = 4;
  BndView view() const { return BndView{rows.p, ptr.p, mid.p, col.p, val.p, n, lanes}; }
};

int pick_lanes(double mean);

void build_bnd(const LocalCsr& oo, const LocalCsr& og, DevBnd& d) {
  BndHost hb;
  bnd_layout(oo, og, hb);
  d.n = (int)hb.rows.size();
  d.lanes = hb.lanes;
  d.rows.upload(hb.rows);
  d.ptr.upload(hb.ptr);
  d.mid.upload(hb.mid);
  d.col.upload(hb.col);
  d.val.upload(hb.val);
  d.skip.upload(hb.skip);
}

// Rows of all parts of one operator merged into one matrix in gid numbering (replicated coarse tail).
// which: PAMG_A_OO (rows/cols level l), PAMG_P_OO (rows l, cols l+1), PAMG_R_OO (rows l+1, cols l).
// A row keeps the order mul! sums it in: own-part columns, then ghost columns.
void merged_block(const Hierarchy& h, int l, int which, LocalCsr& out) {
  const int lr = which == PAMG_R_OO ? l + 1 : l;
  const int lc = which == PAMG_P_OO ? l + 1 : l;
  const int64_t nr = h.levels[lr].n_global, nc = h.levels[lc].n_global;
  out = LocalCsr();
  out.nrows = nr;
  out.ncols = nc;
  out.ptr.assign(nr + 1, 0);
  for (int p = 0; p < h.nparts; ++p) {
    const PartLevel& pl = h.levels[l].parts[p];
    const PartLevel& pr = h.levels[lr].parts[p];
    if (!pl.full || !pr.full || !h.levels[lc].parts[p].full)
      throw std::runtime_error("replicated tail needs every part of its levels: the hierarchy was loaded with a smaller tail_rows");
    const LocalCsr &oo = pl.blk[which], &og = pl.blk[which + 1];
    for (int64_t i = 0; i < pr.n_own; ++i) {
      int64_t cnt = 0;
      if (!oo.ptr.empty()) cnt += oo.ptr[i + 1] - oo.ptr[i];
      if (!og.ptr.empty()) cnt += og.ptr[i + 1] - og.ptr[i];
      out.ptr[pr.own_to_global[i] + 1] = cnt;
    }
  }
  for (int64_t g = 0; g < nr; ++g) out.ptr[g + 1] += out.ptr[g];
  if (out.ptr[nr] > INT32_MAX) throw std::runtime_error("merged tail level exceeds int32 entries (lower tail_rows)");
  out.col.resize(out.ptr[nr]);
  out.val.resize(out.ptr[nr]);
  for (int p = 0; p < h.nparts; ++p) {
    const PartLevel& pl = h.levels[l].parts[p];
    const PartLevel& pr = h.levels[lr].parts[p];
    const PartLevel& pc = h.levels[lc].parts[p];
    const LocalCsr &oo = pl.blk[which], &og = pl.blk[which + 1];
    for (int64_t i = 0; i < pr.n_own; ++i) {
      int64_t q = out.ptr[pr.own_to_global[i]];
      if (!oo.ptr.empty())
        for (int64_t k = oo.ptr[i]; k < oo.ptr[i + 1]; ++k) {
          out.col[q] = (int32_t)pc.own_to_global[oo.col[k]];
          out.val[q++] = oo.val[k];
        }
      if (!og.ptr.empty())
        for (int64_t k = og.ptr[i]; k < og.ptr[i + 1]; ++k) {
          out.col[q] = (int32_t)pc.ghost_to_global[og.col[k]];
          out.val[q++] = og.val[k];
        }
    }
  }
}

// AUTO takes SELL-C-sigma when its padding stores at most this many entries per nonzero
constexpr double SELL_AUTO_MAX_FILL = 1.25;
// AUTO per operator (gpurun kernel sweep, profiles/r01_kernel_sweep.md): A -> SELL (0.29 vs 0.36 ms at 256^3);
// R -> SELL only with enough coarse rows to fill the GPU one thread per row, else CSR-stream (few, long rows);
// P (1-8 entries per row) -> SELL like A once its short rows run as one resident wave of persistent CTAs (0.228 vs 0.268 ms).
// (one thread per row needs >= ~200k rows to fill 148 SMs: at 44k rows x 68 nnz the SELL sweep takes 63 us, CSR-stream 20 us)
constexpr int64_t SELL_AUTO_MIN_ROWS_A = 200000, SELL_AUTO_MIN_ROWS_R = 65536;

int pick_lanes(double mean) {
  if (mean <= 1.5) return 1;
  if (mean <= 3.0) return 2;
  if (mean <= 6.0) return 4;
  if (mean <= 12.0) return 8;
  if (mean <= 24.0) return 16;
  return 32;
}

// fmt: PAMG_FORMAT_* requested for this block (own-ghost blocks are always compressed-row CSR)
void build_csr(const LocalCsr& m, bool compress, DevCsr& d, int lanes_override, int fmt, const pamg_options& o, int which) {
  const int64_t nr = m.nrows;
  std::vector<int32_t> ptr;
  d.listed = compress;
  d.nnz = m.nnz();
  d.stream = false;
  d.nblocks = 0;
  d.sell_rpt = 0;
  d.sell_vi = false;
  d.sell_vi4 = false;
  d.sell_diag = false;
  if (m.ptr.empty()) {  // absent block
    d.nrows = compress ? 0 : (int32_t)nr;
    ptr.assign((compress ? 0 : nr) + 1, 0);
    d.ptr.upload(ptr);
    d.col.alloc(16);
    d.val.alloc(16);
    d.rows.alloc(0);
    return;
  }
  if (compress) {
    std::vector<int32_t> rows;
    ptr.push_back(0);
    for (int64_t i = 0; i < nr; ++i)
      if (m.ptr[i + 1] > m.ptr[i]) {
        rows.push_back((int32_t)i);
        ptr.push_back((int32_t)m.ptr[i + 1]);
      }
    d.nrows = (int32_t)rows.size();
    d.rows.upload(rows);
  } else {
    ptr.resize(nr + 1);
    for (int64_t i = 0; i <= nr; ++i) ptr[i] = (int32_t)m.ptr[i];
    d.nrows = (int32_t)nr;
    d.rows.alloc(0);
  }
  const double mean = d.nrows ? (double)d.nnz / d.nrows : 0.0;
  d.lanes = lanes_override > 0 ? lanes_override : pick_lanes(mean);
  // ---- SELL-C-sigma ----
  bool auto_sell = false;
  if (fmt == PAMG_FORMAT_AUTO) {
    if (which == PAMG_A_OO || which == PAMG_P_OO) auto_sell = nr >= SELL_AUTO_MIN_ROWS_A;
    if (which == PAMG_R_OO) auto_sell = nr >= SELL_AUTO_MIN_ROWS_R;
  }
  const bool sell_req = fmt == PAMG_FORMAT_SELL || fmt == PAMG_FORMAT_SELL_DIAG;
  if (!compress && nr > 0 && (sell_req || auto_sell)) {
    const int rpt = (o.sell_rows_per_thread == 1 || o.sell_rows_per_thread == 2) ? o.sell_rows_per_thread : 2;
    // stencil A blocks: implied columns, one index byte per slot (0.117 instead of 0.585 GB per pass over A0 at 256^3); only under AUTO and
    // SELL_DIAG (an explicit SELL keeps the column-stored layouts), and like every value-indexed layout not with PAMG_VALUE_INDEX=0
    const char* ve = getenv("PAMG_VALUE_INDEX");
    DiagHost dh;
    if (which == PAMG_A_OO && fmt != PAMG_FORMAT_SELL && rpt == 2 && !(ve && atoi(ve) == 0) && diag_layout(m, dh, true)) {
      d.sl_dict.upload(dh.dict);
      d.ndict = (int)dh.dict.size();
      d.dg_off.upload(dh.off);
      std::vector<uint32_t> words(dh.idx.size() / 4);
      std::memcpy(words.data(), dh.idx.data(), dh.idx.size());
      d.dg_idx.upload(words);
      d.ndiag = (int)dh.off.size();
      d.nslices4 = (int)dh.nslices;
      d.nslices = 0;
      d.sell_diag = true;
      d.sell_rpt = 2;
      d.sell_perm = false;
      d.sell_sigma = 1;
      d.sell_fill = (double)d.ndiag * (double)nr / (double)d.nnz;
      d.ptr.alloc(1);
      d.col.alloc(16);
      d.val.alloc(16);
      return;
    }
    const int C = 32 * rpt;
    SellHost sh;
    int sigma = o.sell_sigma > 0 ? o.sell_sigma : 1;
    sell_layout(m, C, sigma, sh, false);
    // few distinct values (stencil matrices, their prolongators): value-indexed storage, 5 instead of 12 bytes per entry; up to
    // VI_WIDE_MAX - 1 distinct values (Galerkin matrix of the first coarse level): two index bytes, 6 instead of 12 (128-row layout only)
    bool vi_ok = false, vi_wide = false;
    {
      const char* e = getenv("PAMG_VALUE_INDEX");
      const bool on = rpt == 2 && !(e && atoi(e) == 0);
      vi_ok = on && value_dictionary(m, sh.dict, 255);
      if (on && !vi_ok && !(e && atoi(e) == 1) && o.sell_sigma <= 1)
        vi_wide = value_dictionary(m, sh.dict, VI_WIDE_MAX - 1);  // PAMG_VALUE_INDEX=1: one-byte indices only
    }
    // auto sigma: sort inside windows only when the unsorted padding is large (the permutation costs more than
    // ~20 % padding does: P at 256^3 runs 0.228 ms unsorted with 1.16x fill, 0.240 ms sorted with 1.01x).  A value-indexed
    // block pads with 5-byte entries and pays the same for the permutation: 0.202 ms unsorted (1.41x) vs 0.229 ms sorted
    const double sort_fill = (vi_ok || vi_wide) ? 2.0 : 1.25;
    if (o.sell_sigma <= 0 && sh.fill > sort_fill) {
      SellHost s2;
      sell_layout(m, C, 64 * C, s2, false);
      if (s2.fill < sh.fill - 0.02) sigma = 64 * C;
      sh.fill = std::min(sh.fill, s2.fill);
    }
    const bool take = sell_req || sh.fill <= std::max(SELL_AUTO_MAX_FILL, sort_fill);
    if (take) {
      sell_layout(m, C, sigma, sh, true);
      d.sl_off.upload(sh.off);
      d.sl_col.upload(sh.col);
      d.sl_val.upload(sh.val);
      d.sell_vi = false;
      d.sell_vi4 = false;
      if (vi_ok) {
        sell_value_index(sh, 1);
        d.sl_vidx.upload(sh.vidx);
        d.sell_vi = true;
      }
      if (vi_ok || vi_wide) {
        d.ndict = (int)sh.dict.size();
        d.sl_dict.upload(sh.dict);
        // four interleaved rows per lane (k_spmv_sell_vi4): a second, 128-row slicing.  Sorted rows keep the two-rows-per-lane kernel.
        if (!sh.permuted) {
          SellHost s4;
          s4.dict = sh.dict;
          sell_layout(m, 128, 1, s4, true, 4);
          d.vi4_ib = vi_ok ? 1 : 2;
          sell_value_index(s4, d.vi4_ib);
          d.v4_off.upload(s4.off);
          d.v4_col.upload(s4.col);
          d.v4_idx.upload(s4.vidx);
          d.nslices4 = (int)s4.off.size() - 1;
          d.sell_vi4 = true;
        }
      }
      d.sell_perm = sh.permuted;
      if (sh.permuted) d.sl_perm.upload(sh.perm);
      d.nslices = (int)sh.off.size() - 1;
      d.sell_rpt = rpt;
      d.sell_sigma = sigma;
      d.sell_fill = sh.fill;
      d.ptr.alloc(1);
      d.col.alloc(16);
      d.val.alloc(16);
      return;
    }
  }
  d.ptr.upload(ptr);
  {  // pad to a multiple of 4 entries (+8) with zeros: the stream kernel reads whole 128-bit groups
    const size_t padded = (m.col.size() + 3) / 4 * 4 + 8;
    std::vector<int32_t> col(m.col);
    std::vector<double> val(m.val);
    col.resize(padded, 0);
    val.resize(padded, 0.0);
    d.col.upload(col);
    d.val.upload(val);
  }
  if (!compress && nr > 0 && fmt != PAMG_FORMAT_CSR) {
    // greedy row blocks: <= S_ROWS rows and <= S_CAP - 3 entries (so the 4-aligned window fits)
    std::vector<std::pair<int32_t, int32_t>> hb;
    const bool ok = stream_row_blocks(m, S_ROWS, S_CAP - 3, hb);
    std::vector<int2> blk;
    for (auto& e : hb) blk.push_back(make_int2(e.first, e.second));
    if (ok) {
      d.nblocks = (int)blk.size() - 1;
      d.blk.upload(blk);
      d.stream = true;
    }
  }
}

// byte offsets inside a part's peer-visible arena; computable by every process for every part
struct ArenaLayout {
  std::vector<size_t> ghost, flags, asm_stage, asm_flags;
  size_t coarse = 0, coarse_flags = 0, red = 0, red_flags = 0, total = 0;
  // a part's arena holds kmax copies of this layout, column j at j * col_stride; the word at `capacity` (behind column 0's
  // layout) is the kmax its owner allocated, checked by every process at connect
  size_t capacity = 0, col_stride = 0;
};

// First level of the replicated coarse tail: levels [tail, L) are merged over all parts and run by every
// GPU alone (coarse-level agglomeration).  Decided from replicated metadata, so every process agrees.
int tail_level_of(const Hierarchy& h) {
  const int L = (int)h.levels.size();
  if (L <= 1) return 0;
  int64_t tail_rows = h.opts.tail_rows;
  if (const char* e = getenv("PAMG_TAIL_ROWS")) tail_rows = std::min<int64_t>(tail_rows, atoll(e));  // experiments: only lowering is safe
  if (h.nparts == 1 || tail_rows <= 0) return L - 1;
  for (int l = 1; l < L; ++l)
    if (h.levels[l].n_global <= tail_rows) return l;
  return L - 1;
}

ArenaLayout arena_layout(const Hierarchy& h, int part) {
  ArenaLayout a;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + std::max<size_t>(bytes, 8), 256);
    return o;
  };
  for (const Level& lev : h.levels) {
    const PartLevel& pl = lev.parts[part];
    a.ghost.push_back(take(2 * (size_t)pl.n_ghost * sizeof(double)));
    a.flags.push_back(take(pl.recv.size() * sizeof(uint32_t)));
    a.asm_stage.push_back(take(2 * (size_t)pl.n_send_entries() * sizeof(double)));
    a.asm_flags.push_back(take(pl.send.size() * sizeof(uint32_t)));
  }
  a.coarse = take(2 * (size_t)h.levels[tail_level_of(h)].n_global * sizeof(double));
  a.coarse_flags = take((size_t)h.nparts * sizeof(uint32_t));
  a.red = take(2 * (size_t)h.nparts * RED_W * sizeof(double));
  a.red_flags = take((size_t)h.nparts * sizeof(uint32_t));
  a.total = off;
  a.capacity = take(sizeof(int32_t));
  a.col_stride = off;
  return a;
}

struct LevelDev {
  int64_t n_own = 0, n_ghost = 0;
  DevCsr blk[6];      // own-own blocks at even indices (own-ghost blocks live in `bnd`)
  DevBnd bnd[3];      // boundary rows of A, P, R
  DBuf<double> w;     // smoother weight: w/a_ii (Jacobi), 1/l1-diag (l1), 1/(theta a_ii) (Chebyshev zero-guess step)
  DBuf<double> dinv;  // 1/a_ii (Chebyshev)
  // per right-hand side: work vectors and the halo staging of that column's arena copy
  struct Col {
    DBuf<double> x, x2, b, t, d, d2;
    double* xstart = nullptr;
    HaloRecv hr{};
    DBuf<SendNbr> send_nbrs;
  };
  std::unique_ptr<Col[]> cols;
  // Views of the BOUND column's buffers (Engine::Impl::bind).  Read them only after selecting the column: Impl::S(slot) (or LV(slot,
  // l)) binds the slot's column; Impl::P(i) does not, so after P(i) these still show whichever column was bound last.
  DView<double> x, x2, b, t, d, d2;
  DBuf<int32_t> send_idx;
  DView<SendNbr> send_nbrs;
  int n_send = 0, n_send_nbrs = 0, n_recv_nbrs = 0;
  HaloRecv hr{};
  // assemble! plan
  DBuf<AsmSendNbr> asm_nbrs;
  DBuf<int32_t> asm_rows, asm_ptr, asm_src;
  int asm_nrows = 0;
  const double* asm_stage = nullptr;
  const uint32_t* asm_flags = nullptr;
  double* xstart = nullptr;  // buffer the zero-guess first sweep is written to (so the V-cycle ends in x)
};

struct Status {  // host mirror of what we read back
  DevState st;
};

}  // namespace

struct PartDev {
  int part = -1, device = 0;
  cudaStream_t stream = nullptr;
  std::vector<std::unique_ptr<LevelDev>> lev;
  std::vector<std::unique_ptr<LevelDev>> tlev;  // merged (replicated) levels [tail_level, L), null below
  ArenaLayout lay;
  char* arena = nullptr;
  // per right-hand side: solve state, Krylov vectors and the all-reduce / coarse-gather wiring of that column's arena copy
  struct Col {
    DBuf<DevState> st;
    DBuf<double> partials, xsol, p, q, bsave, hist, rprev;  // rprev: r_k of flexible CG (allocated on first use)
    int hist_cap = 0;
    DBuf<RedPub> red_pubs;
    RedCtx rc{};
    DBuf<CoarsePub> coarse_pubs;
  };
  std::unique_ptr<Col[]> cols;
  // views of the BOUND column's state: valid for a slot only after Impl::S(slot) (see LevelDev)
  char* carena = nullptr;
  DView<DevState> st;
  DView<double> partials, xsol, p, q, bsave, hist, rprev;
  RedCtx rc{};
  DView<CoarsePub> coarse_pubs;
  int partials_cap = 0;
  DBuf<double> inv;
  DBuf<int64_t> own_gid_T, ghost_gid_T;
  DBuf<double> scratch4;
  DBuf<double> io_local;  // own+ghost staging for consistent!/assemble!
  DBuf<double> gm_basis;  // FGMRES: V_0..V_m then Z_0..Z_{m-1}, own length each (allocated on first use)
  DBuf<double> gm_h;      // FGMRES: one Hessenberg column (m + 2 doubles), written by k_gs_sub / k_gs_norm
  int gm_restart = 0;
  bool gm_precond = false;
  DBuf<unsigned long long> trace;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

struct Engine::Impl {
  Hierarchy* h = nullptr;
  int nparts = 0, L = 0;
  int tail_level = 0;      // levels >= tail_level run replicated (merged over all parts) on every GPU
  bool tail_mode = false;  // enqueue_* address the merged levels
  LevelDev& LV(PartDev& pd, int l) { return tail_mode ? *pd.tlev[l] : *pd.lev[l]; }
  LevelDev& LV(size_t s, int l) { return LV(S(s), l); }  // slot s (binds its column)
  std::vector<std::unique_ptr<PartDev>> parts;         // local parts
  std::vector<int> local_index;                        // part -> index in parts or -1
  std::vector<char*> arena_of;                         // part -> arena base as seen from this process
  std::vector<cudaIpcMemHandle_t> ipc;                 // part -> handle (remote parts)
  std::vector<char> have_ipc;
  std::vector<void*> ipc_opened;
  std::map<int, cudaStream_t> stream_of_device;
  bool connected = false;
  bool fused_halo = false;  // every local part has a GPU of its own: halo roles run inside the consuming kernel
  bool fold_check = false;  // the convergence check runs inside k_update_xr / k_pcg_init (every local part alone on its GPU)
  int64_t launches = 0;
  bool counting = true;
  // exchange needed per level/operator (decided on global metadata so every part agrees)
  std::vector<char> need_halo_A, need_halo_R, need_halo_P;
  // graphs (one per distinct stream)
  std::vector<cudaGraphExec_t> g_iter, g_vcycle, g_vcycle_multi;
  std::vector<cudaStream_t> g_streams;
  int64_t g_iter_nodes = 0, g_vcycle_nodes = 0, g_vcycle_multi_nodes = 0;
  int g_iter_mode = -1;  // mode the iteration graph was captured for: 0 plain CG, 1 PCG, 2 flexible PCG
  int g_iter_k = 0;      // columns it was captured for (0: the single-column solve), likewise for g_vcycle_multi
  int g_vcycle_multi_k = 0;
  double* flush_buf = nullptr;
  size_t flush_n = 0;
  pamg_stats stats{};
  HostStat* hstat_base = nullptr;  // pinned, device-mapped rings (HS_RING per column) written by k_check of the first local part
  HostStat* hstat = nullptr;       // the bound column's ring
  bool rhs_loaded = false;
  // right-hand sides: kmax columns of per-solve state exist; `cols` are the ones the enqueue_* functions run over (slot s = column
  // cols[s / nparts_local], part s % nparts_local), {0} outside multi-column calls, which also set `multi` (split halo launches)
  int kmax = 1;
  std::vector<int> cols{0};
  bool multi = false;
  int bound = -1;
  size_t nslots() const { return cols.size() * parts.size(); }
  int col_of(size_t s) const { return cols[s / parts.size()]; }
  PartDev& S(size_t s) {
    bind(col_of(s));
    return *parts[s % parts.size()];
  }
  // point the views of every part and level at column c's buffers
  void bind(int c, bool force = false) {
    if (c == bound && !force) return;
    bound = c;
    auto bind_level = [c](LevelDev& ld) {
      LevelDev::Col& lc = ld.cols[c];
      ld.x = lc.x;
      ld.x2 = lc.x2;
      ld.b = lc.b;
      ld.t = lc.t;
      ld.d = lc.d;
      ld.d2 = lc.d2;
      ld.xstart = lc.xstart;
      ld.hr = lc.hr;
      ld.send_nbrs = lc.send_nbrs;
    };
    for (auto& up : parts) {
      PartDev& pd = *up;
      PartDev::Col& pc = pd.cols[c];
      pd.carena = pd.arena + (size_t)c * pd.lay.col_stride;
      pd.st = pc.st;
      pd.partials = pc.partials;
      pd.xsol = pc.xsol;
      pd.p = pc.p;
      pd.q = pc.q;
      pd.bsave = pc.bsave;
      pd.hist = pc.hist;
      pd.rprev = pc.rprev;
      pd.rc = pc.rc;
      pd.coarse_pubs = pc.coarse_pubs;
      for (auto& ld : pd.lev) bind_level(*ld);
      for (auto& ld : pd.tlev)
        if (ld) bind_level(*ld);
    }
    hstat = hstat_base + (size_t)c * HS_RING;
  }

  ~Impl();
  PartDev& P(int i) { return *parts[i]; }
  void set_dev(const PartDev& p) { CK(cudaSetDevice(p.device)); }
  // fine-grained blocks (hardware schedules them dynamically, no tail); capped at MAX_GRID because
  // kernels with a fused reduction write one partial per block
  static constexpr int MAX_GRID = 16384;
  int grid_for(int64_t work_items, int items_per_block) const {
    int64_t g = (work_items + items_per_block - 1) / items_per_block;
    return (int)std::max<int64_t>(1, std::min<int64_t>(g, MAX_GRID));
  }
  // kernels with a fused reduction: one fence + ticket per CTA, so keep the CTA count small
  int grid_red(int64_t work_items) const {
    return (int)std::max<int64_t>(1, std::min<int64_t>((work_items + BLOCK - 1) / BLOCK, RED_GRID));
  }
  std::vector<std::string> names;  // kernel names in launch order while `naming` (graph capture of one PCG iteration)
  bool naming = false;
  void note_launch(const char* name = "kernel") {
    if (counting) ++launches;
    if (naming) names.push_back(name);
  }
};

Engine::Impl::~Impl() {
  for (auto g : g_iter) cudaGraphExecDestroy(g);
  for (auto g : g_vcycle) cudaGraphExecDestroy(g);
  for (auto g : g_vcycle_multi) cudaGraphExecDestroy(g);
  if (hstat_base) cudaFreeHost(hstat_base);
  for (auto& up : parts) {
    cudaSetDevice(up->device);
    if (up->ev0) cudaEventDestroy(up->ev0);
    if (up->ev1) cudaEventDestroy(up->ev1);
    if (up->arena) cudaFree(up->arena);
  }
  if (flush_buf) cudaFree(flush_buf);
  for (void* p : ipc_opened) cudaIpcCloseMemHandle(p);
  parts.clear();
  for (auto& kv : stream_of_device) {
    cudaSetDevice(kv.first);
    cudaStreamDestroy(kv.second);
  }
}

// ---------------------------------------------------------------------------------------------
// kernel dispatch
// ---------------------------------------------------------------------------------------------
namespace {

// CTAs of `kernel` that are resident at once on the current device (148 SMs x occupancy): the grid of a
// kernel with a fused reduction, so that it runs as exactly one wave of persistent CTAs
int resident_ctas(const void* kernel, size_t dyn_smem = 0) {
  static std::map<std::tuple<int, const void*, size_t>, int> cache;
  int dev = 0;
  cudaGetDevice(&dev);
  auto key = std::make_tuple(dev, kernel, dyn_smem);
  auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  int per_sm = 0, sms = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, BLOCK, dyn_smem) != cudaSuccess) per_sm = 2;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
  const int r = std::max(1, per_sm * sms);
  cache[key] = r;
  return r;
}

struct LaunchArgs {  // what every SpMV-family launch shares
  int grid;            // boundary launch: the grid; main launches: natural number of main CTAs
  bool bounded;        // main launches: cap the main CTAs at one resident wave (fused reductions)
  cudaStream_t s;
  const double* x;
  EpiArgs a;
  DevState* st;
  FusedHalo fh;
  double* partials;
  RedCtx rc;
  int publish, slot;   // fused dot: publish = 1 total goes to every part, 0 a boundary launch completes it
};

// The kernel an operation runs, decided once from its block (and long_rows, see launch_stream); the launch and the trace name both follow
// from it.
enum class SpmvKernel { SellDiag, SellVi, SellVi16, SellVi2, Sell, Stream, StreamLong, Csr };
// sell-vi = four rows per lane (one-byte indices), sell-vi16 = the same with two-byte indices, sell-vi2 = two rows per lane (sorted rows)
const char* const SPMV_KERNEL_NAMES[] = {"sell-diag", "sell-vi", "sell-vi16", "sell-vi2", "sell", "stream", "stream-long", "csr"};

SpmvKernel spmv_kernel(const DevCsr& m, bool long_rows) {
  if (m.sell_diag) return SpmvKernel::SellDiag;
  if (m.sell_vi4) return m.vi4_ib == 2 ? SpmvKernel::SellVi16 : SpmvKernel::SellVi;
  if (m.sell_vi) return SpmvKernel::SellVi2;
  if (m.sell_rpt) return SpmvKernel::Sell;
  if (m.stream) return long_rows ? SpmvKernel::StreamLong : SpmvKernel::Stream;
  return SpmvKernel::Csr;
}

int main_grid(const LaunchArgs& L, const void* kernel, size_t dyn_smem = 0) {
  int n_main = L.grid;
  if (L.bounded) n_main = std::min(n_main, std::min(resident_ctas(kernel, dyn_smem), RED_GRID));
  return L.fh.n_pack + std::max(n_main, 1) + L.fh.n_bnd;
}

// MODE x DOT dispatch; F(mode_tag, dot_tag) launches one instantiation
template <class F>
void dispatch_mode(int mode, bool dot, F&& f) {
#define PAMG_M(MD, DT) \
  case MD:             \
    f(std::integral_constant<int, MD>{}, std::integral_constant<bool, DT>{}); \
    break;
  if (dot) {
    switch (mode) {
      PAMG_M(M_MUL, true)
      PAMG_M(M_JACOBI, true)
      default:
        throw std::runtime_error("fused dot only on MUL/JACOBI");
    }
  } else {
    switch (mode) {
      PAMG_M(M_MUL, false)
      PAMG_M(M_RESID, false)
      PAMG_M(M_JACOBI, false)
      PAMG_M(M_ADD, false)
      PAMG_M(M_RESTRICT, false)
      PAMG_M(M_CHEB, false)
      default:
        throw std::runtime_error("bad mode");
    }
  }
#undef PAMG_M
}

void launch_csr(int mode, bool dot, int lanes, CsrView A, const LaunchArgs& L) {
  dispatch_mode(mode, dot, [&](auto md, auto dt) {
    constexpr int MD = decltype(md)::value;
    constexpr bool DT = decltype(dt)::value;
#define PAMG_L(LN)                                                                                                         \
  case LN:                                                                                                                 \
    k_spmv<LN, MD, DT><<<main_grid(L, (const void*)k_spmv<LN, MD, DT>), BLOCK, 0, L.s>>>(A, L.x, L.a, L.st, L.fh, L.partials, L.rc, \
                                                                                        L.publish, L.slot);               \
    break;
    switch (lanes) {
      PAMG_L(1)
      PAMG_L(2)
      PAMG_L(4)
      PAMG_L(8)
      PAMG_L(16)
      PAMG_L(32)
      default:
        throw std::runtime_error("bad lanes_per_row");
    }
#undef PAMG_L
  });
}

// long_rows: mean row length >= 48 -> the phase-B variant with 16 lanes per row (kernels.cuh k_spmv_stream LONG)
void launch_stream(int mode, bool dot, bool long_rows, StreamView A, const LaunchArgs& L) {
  dispatch_mode(mode, dot, [&](auto md, auto dt) {
    constexpr int MD = decltype(md)::value;
    constexpr bool DT = decltype(dt)::value;
    using Kern = void (*)(StreamView, const double*, EpiArgs, DevState*, FusedHalo, double*, RedCtx, int, int);
    Kern k = k_spmv_stream<MD, DT, false>;
    if constexpr (!DT) {
      if (long_rows) k = k_spmv_stream<MD, false, true>;
    }
    k<<<main_grid(L, (const void*)k), BLOCK, 0, L.s>>>(A, L.x, L.a, L.st, L.fh, L.partials, L.rc, L.publish, L.slot);
  });
}

void launch_sell(int mode, bool dot, int rpt, SellView A, const LaunchArgs& L) {
  dispatch_mode(mode, dot, [&](auto md, auto dt) {
    constexpr int MD = decltype(md)::value;
    constexpr bool DT = decltype(dt)::value;
    using Kern = void (*)(SellView, const double*, EpiArgs, DevState*, FusedHalo, double*, RedCtx, int, int);
    Kern k = rpt == 2 ? (Kern)k_spmv_sell<2, MD, DT> : (Kern)k_spmv_sell<1, MD, DT>;
    k<<<main_grid(L, (const void*)k), BLOCK, 0, L.s>>>(A, L.x, L.a, L.st, L.fh, L.partials, L.rc, L.publish, L.slot);
  });
}

// value-indexed, two rows per lane (blocks with sorted rows)
void launch_sell_vi(int mode, bool dot, const SellViView& A, const LaunchArgs& L) {
  dispatch_mode(mode, dot, [&](auto md, auto dt) {
    constexpr int MD = decltype(md)::value;
    constexpr bool DT = decltype(dt)::value;
    auto k = k_spmv_sell_vi<MD, DT>;
    k<<<main_grid(L, (const void*)k), BLOCK, 0, L.s>>>(A, L.x, L.a, L.st, L.fh, L.partials, L.rc, L.publish, L.slot);
  });
}

// value-indexed, four rows per lane with ib index bytes per entry.  A launch bounded to one resident wave takes the look-ahead, and in the
// one-byte form U = 2 at 4 CTAs/SM (kernels.cuh k_spmv_sell_vi4).
void launch_sell_vi4(int mode, bool dot, int ib, const SellViView& A, const LaunchArgs& L) {
  dispatch_mode(mode, dot, [&](auto md, auto dt) {
    constexpr int MD = decltype(md)::value;
    constexpr bool DT = decltype(dt)::value;
    using Kern = void (*)(SellViView, const double*, EpiArgs, DevState*, FusedHalo, double*, RedCtx, int, int);
    const Kern by_ib_bounded[2][2] = {{k_spmv_sell_vi4<MD, DT, 1>, k_spmv_sell_vi4<MD, DT, 1, 2, 4, 1>},
                                      {k_spmv_sell_vi4<MD, DT, 2>, k_spmv_sell_vi4<MD, DT, 2, 4, 3, 1>}};
    const Kern k = by_ib_bounded[ib == 2][L.bounded];
    const size_t dyn = (size_t)A.ndict * sizeof(double);  // the dictionary lives in dynamic shared memory
    k<<<main_grid(L, (const void*)k, dyn), BLOCK, dyn, L.s>>>(A, L.x, L.a, L.st, L.fh, L.partials, L.rc, L.publish, L.slot);
  });
}

// grid as for the vi4 kernel it replaces (same occupancy): the same resident CTAs, so the fused dots add in the same order
void launch_sell_diag(int mode, bool dot, const SellDiagView& A, const LaunchArgs& L) {
  dispatch_mode(mode, dot, [&](auto md, auto dt) {
    constexpr int MD = decltype(md)::value;
    constexpr bool DT = decltype(dt)::value;
    auto k = k_spmv_sell_diag<MD, DT>;
    k<<<main_grid(L, (const void*)k), BLOCK, 0, L.s>>>(A, L.x, L.a, L.st, L.fh, L.partials, L.rc, L.publish, L.slot);
  });
}

// k-wide form of the block's kernel for K columns (multi-column calls, main role only).  The grid is the one the single kernel would
// get for this launch, so every column sees the same slices per CTA and the same fused-dot partials as on its own.
//
// Width of the launch for the next g (>= 1) columns of one block: 2 or 4 (one k-wide launch; g = 3 runs K = 4 with one column absent)
// or 1 (the single kernel for one column).  Chosen per block class from the B200 measurements of DESIGN §4.9
// (profiles/r05_multi_rhs.json; L2 flushed, k-wide launch against k single launches): the k-wide forms hold 2 CTAs per SM against the
// single kernels' 3-4, and where that loses the class keeps its single launches:
//   implied-column A (k_spmv_sell_diag): K = 2 loses in every mode (1.17x the time of two single launches for the Jacobi sweep); K = 4
//     wins for the Jacobi sweep (0.93x), the residual and the SpMV + p.q (0.83x) but loses for the Jacobi sweep + r.z (1.07x);
//   value-indexed P (prolongation, 1-8 entries per row): 1.04-1.24x at K = 2 and 4 on the Poisson and jump-coefficient hierarchies;
//   value-indexed A and R (elasticity A0, level-1 A, restriction): 0.61-0.97x at K = 2 and 4 in every mode measured.
int multi_width(SpmvKernel k, int which, int mode, bool dot, int g) {
  if (g < 2) return 1;
  if (k == SpmvKernel::SellDiag) return (g >= 3 && !(mode == M_JACOBI && dot)) ? 4 : 1;
  if ((k == SpmvKernel::SellVi || k == SpmvKernel::SellVi16) && which != PAMG_P_OO) return g == 2 ? 2 : 4;
  return 1;
}

template <int K>
void launch_multi(SpmvKernel kern, const DevCsr& m, int mode, bool dot, const LaunchArgs& L, const MultiCols<K>& mc) {
  dispatch_mode(mode, dot, [&](auto md, auto dt) {
    constexpr int MD = decltype(md)::value;
    constexpr bool DT = decltype(dt)::value;
    if (kern == SpmvKernel::SellDiag) {
      const int grid = main_grid(L, (const void*)k_spmv_sell_diag<MD, DT>);
      k_spmv_sell_diag_multi<MD, DT, K><<<grid, BLOCK, 0, L.s>>>(m.diagview(), mc, L.fh, L.publish, L.slot);
      return;
    }
    using Kern = void (*)(SellViView, const double*, EpiArgs, DevState*, FusedHalo, double*, RedCtx, int, int);
    const Kern by_ib_bounded[2][2] = {{k_spmv_sell_vi4<MD, DT, 1>, k_spmv_sell_vi4<MD, DT, 1, 2, 4, 1>},
                                      {k_spmv_sell_vi4<MD, DT, 2>, k_spmv_sell_vi4<MD, DT, 2, 4, 3, 1>}};
    const size_t dyn = (size_t)m.ndict * sizeof(double);
    const int grid = main_grid(L, (const void*)by_ib_bounded[m.vi4_ib == 2][L.bounded], dyn);
    if (m.vi4_ib == 2)
      k_spmv_sell_vi4_multi<MD, DT, 2, K><<<grid, BLOCK, dyn, L.s>>>(m.vi4view(), mc, L.fh, L.publish, L.slot);
    else
      k_spmv_sell_vi4_multi<MD, DT, 1, K><<<grid, BLOCK, dyn, L.s>>>(m.vi4view(), mc, L.fh, L.publish, L.slot);
  });
}

void launch_boundary(int mode, bool dot, const LaunchArgs& L) {
  dispatch_mode(mode, dot, [&](auto md, auto dt) {
    k_boundary<decltype(md)::value, decltype(dt)::value><<<L.grid, BLOCK, 0, L.s>>>(L.x, L.a, L.st, L.fh, L.partials, L.rc, L.slot);
  });
}

}  // namespace

// One SpMV-family operation over all local parts: consistent!(xin) + own rows of the operator.
// which: PAMG_A_OO / PAMG_P_OO / PAMG_R_OO (the matching *_OG is implied).
// row_level: level whose LevelDev holds the blocks; halo_level: level of the column partition.
struct OpSpec {
  int row_level, which, halo_level, mode;
  bool dot = false;
  int slot = 0;
  bool coarse_ghosts_local = false;  // P at the coarsest level: ghost values were computed locally (parity 0)
};

void Engine::enqueue_op(const OpSpec& op, const std::vector<const double*>& xin, const std::vector<EpiArgs>& epi) {
  Impl& I = *impl;
  const int l = op.row_level;
  bool need;
  if (op.which == PAMG_A_OO)
    need = I.need_halo_A[op.halo_level];
  else if (op.which == PAMG_R_OO)
    need = I.need_halo_R[l];
  else
    need = I.need_halo_P[l];
  if (I.tail_mode) need = false;  // merged levels: every column is an own column
  const bool exchange = need && !op.coarse_ghosts_local;
  const bool fused = I.fused_halo && !I.multi;  // multi-column calls: split launches on every layout
  const int wsel = op.which / 2;  // 0 A, 1 P, 2 R
  const size_t np = I.parts.size(), ns = I.nslots();

  auto halo_args = [&](PartDev& pd, bool with_pack, bool with_bnd) {
    LevelDev& ld = I.LV(pd, l);
    LevelDev& hl = I.LV(pd, op.halo_level);
    FusedHalo fh{};
    fh.level = op.halo_level;
    fh.fixed_parity = op.coarse_ghosts_local ? 0 : -1;
    fh.fused = fused ? 1 : 0;
    // boundary CTAs ahead of a SMALL main role (their latency is all there is), behind a large one (ahead of it
    // they would hold resident-CTA slots while they spin: 256^3 on 4 GPUs 17.1 -> 15.9 ms)
    fh.bnd_first = ld.blk[op.which].nnz < 4000000 ? 1 : 0;
    fh.skip = need ? ld.bnd[wsel].skip.p : nullptr;
    if (ld.bnd[wsel].n == 0) fh.skip = nullptr;
    if (with_pack) {
      fh.n_pack = std::max(1, std::min(2 * 148, (hl.n_send + BLOCK - 1) / BLOCK));  // one value per thread: no serial store chain
      fh.n_send = hl.n_send;
      fh.n_nbrs = hl.n_send_nbrs;
      fh.send_idx = hl.send_idx.p;
      fh.nbrs = hl.send_nbrs.p;
    }
    if (with_bnd) {
      const DevBnd& b = ld.bnd[wsel];
      const int rpb = BLOCK / b.lanes;
      fh.n_bnd = std::max(1, std::min(4 * 148, (b.n + rpb - 1) / rpb));
      fh.B = b.view();
      fh.hr = hl.hr;
    }
    return fh;
  };
  auto launch_name = [&](SpmvKernel kern, int width, const FusedHalo& fh) {
    static const char* MODES[] = {"mul", "resid", "jacobi", "add", "restrict", "cheb"};
    static const char* OPS[] = {"A", "P", "R"};
    I.names.push_back(std::string(SPMV_KERNEL_NAMES[(int)kern]) + (width > 1 ? " x" + std::to_string(width) : "") + " " + MODES[op.mode] +
                      (op.dot ? "+dot " : " ") + OPS[wsel] + std::to_string(l) + (I.tail_mode ? " tail" : "") + (fh.n_pack ? " +pack" : "") +
                      (fh.n_bnd ? " +bnd" : ""));
    I.naming = false;
    I.note_launch();
    I.naming = true;
  };
  // the launch arguments of slot s (its column must be bound)
  auto main_args = [&](PartDev& pd, size_t s, const FusedHalo& fh, int publish, SpmvKernel* kern) {
    LevelDev& ld = I.LV(pd, l);
    const DevCsr& m = ld.blk[op.which];
    // persistent main role: one resident wave of CTAs striding over the slices / row blocks.  Measured on
    // B200 (256^3): SELL Jacobi sweep 0.316 ms persistent vs 0.344 ms with one CTA per 8 slices.
    // Long rows (level >= 1, 30+ entries per row) lose 10 % that way: they keep one CTA per 8 slices.
    const double mean_nnz = m.nrows ? (double)m.nnz / m.nrows : 0.0;
    const bool bounded = m.sell_rpt && mean_nnz <= 12.0;
    *kern = spmv_kernel(m, mean_nnz >= 48.0 && !op.dot);
    LaunchArgs L{0, bounded || op.dot, pd.stream, xin[s], epi[s], pd.st.p, fh, pd.partials.p, pd.rc, publish, op.slot};
    L.fh.v = xin[s];
    int n_main;
    if (m.sell_diag || m.sell_vi4) {
      n_main = (m.nslices4 + BLOCK / 32 - 1) / (BLOCK / 32);
    } else if (m.sell_rpt) {
      n_main = (m.nslices + BLOCK / 32 - 1) / (BLOCK / 32);
    } else if (m.stream) {
      n_main = m.nblocks;
    } else {
      n_main = I.grid_for(m.nrows, (BLOCK / m.lanes) * 4);
    }
    L.grid = std::max(n_main, 1);
    return L;
  };
  auto launch_main = [&](PartDev& pd, size_t s, const FusedHalo& fh, int publish) {
    LevelDev& ld = I.LV(pd, l);
    const DevCsr& m = ld.blk[op.which];
    SpmvKernel kern;
    const LaunchArgs L = main_args(pd, s, fh, publish, &kern);
    switch (kern) {
      case SpmvKernel::SellDiag: launch_sell_diag(op.mode, op.dot, m.diagview(), L); break;
      case SpmvKernel::SellVi:
      case SpmvKernel::SellVi16: launch_sell_vi4(op.mode, op.dot, m.vi4_ib, m.vi4view(), L); break;
      case SpmvKernel::SellVi2: launch_sell_vi(op.mode, op.dot, m.viview(), L); break;
      case SpmvKernel::Sell: launch_sell(op.mode, op.dot, m.sell_rpt, m.slview(), L); break;
      case SpmvKernel::Stream:
      case SpmvKernel::StreamLong: launch_stream(op.mode, op.dot, kern == SpmvKernel::StreamLong, m.sview(), L); break;
      case SpmvKernel::Csr: launch_csr(op.mode, op.dot, m.lanes, m.view(), L); break;
    }
    if (I.naming)
      launch_name(kern, 1, fh);
    else
      I.note_launch();
  };
  // K columns of part i in one k-wide launch: slots ss[0..n), n <= K (the rest absent)
  auto launch_group = [&](auto kc, size_t i, const size_t* ss, int n, const FusedHalo& fh, int publish) {
    constexpr int K = decltype(kc)::value;
    MultiCols<K> mc{};
    LaunchArgs L{};
    SpmvKernel kern = SpmvKernel::Csr;
    for (int c = 0; c < n; ++c) {
      PartDev& pd = I.S(ss[c]);
      const LaunchArgs Lc = main_args(pd, ss[c], fh, publish, &kern);
      if (c == 0) L = Lc;
      mc.x[c] = Lc.x;
      mc.a[c] = Lc.a;
      mc.st[c] = Lc.st;
      mc.partials[c] = Lc.partials;
      mc.rc[c] = Lc.rc;
    }
    launch_multi<K>(kern, I.LV(I.P(i), l).blk[op.which], op.mode, op.dot, L, mc);
    if (I.naming)
      launch_name(kern, n, fh);
    else
      I.note_launch();
  };

  if (fused) {  // one launch per part: pack + main + boundary roles
    for (size_t i = 0; i < np; ++i) {
      PartDev& pd = I.P(i);
      LevelDev& hl = I.LV(pd, op.halo_level);
      const bool nbrs = hl.n_recv_nbrs > 0 || hl.n_send_nbrs > 0;
      I.set_dev(pd);
      const FusedHalo fh = halo_args(pd, exchange && nbrs, need && nbrs);
      launch_main(pd, i, fh, 1);
    }
    CK(cudaGetLastError());
    return;
  }
  // split: three phases over all parts so that no kernel waits for a later kernel of its own stream
  // phase 1: producers (never wait)
  if (exchange)
    for (size_t s = 0; s < ns; ++s) {
      PartDev& pd = I.S(s);
      LevelDev& hl = I.LV(pd, op.halo_level);
      if (hl.n_send_nbrs == 0 && hl.n_recv_nbrs == 0) continue;
      I.set_dev(pd);
      k_halo_pack<<<I.grid_for(hl.n_send, BLOCK * 4), BLOCK, 0, pd.stream>>>(xin[s], hl.send_idx.p, hl.n_send, hl.send_nbrs.p,
                                                                             hl.n_send_nbrs, pd.st.p, op.halo_level);
      I.note_launch("k_halo_pack");
    }
  // phase 2: all rows of the own-own block (boundary rows are computed but not stored).  Several columns of a block whose class
  // takes a k-wide launch (multi_width) share launches of up to four columns; the others run the single kernel per column.
  // fh, bnd_follows and the kernel depend on the part only (matrices, boundary-row marks, halo plan), not on the bound column:
  // every per-column argument is taken after I.S(slot) in main_args.
  const size_t nc = I.cols.size();
  for (size_t i = 0; i < np; ++i) {
    PartDev& pd = I.P(i);
    LevelDev& hl = I.LV(pd, op.halo_level);
    const bool bnd_follows = need && hl.n_recv_nbrs > 0;
    I.set_dev(pd);
    const FusedHalo fh = halo_args(pd, false, false);
    const SpmvKernel kern = spmv_kernel(I.LV(pd, l).blk[op.which], false);
    for (size_t c0 = 0; c0 < nc;) {
      const int K = multi_width(kern, op.which, op.mode, op.dot, (int)std::min<size_t>(4, nc - c0));
      const int g = std::min<int>(K, (int)(nc - c0));
      size_t ss[4];
      for (int c = 0; c < g; ++c) ss[c] = (c0 + c) * np + i;
      if (K == 1) {
        launch_main(I.S(ss[0]), ss[0], fh, bnd_follows ? 0 : 1);
      } else if (K == 2) {
        launch_group(std::integral_constant<int, 2>{}, i, ss, g, fh, bnd_follows ? 0 : 1);
      } else {
        launch_group(std::integral_constant<int, 4>{}, i, ss, g, fh, bnd_follows ? 0 : 1);
      }
      c0 += g;
    }
  }
  // phase 3: boundary rows (consumers: wait for the neighbours' flags)
  if (need)
    for (size_t s = 0; s < ns; ++s) {
      PartDev& pd = I.S(s);
      LevelDev& hl = I.LV(pd, op.halo_level);
      if (hl.n_recv_nbrs == 0) continue;
      I.set_dev(pd);
      const FusedHalo fh = halo_args(pd, false, true);
      LaunchArgs L{fh.n_bnd, false, pd.stream, xin[s], epi[s], pd.st.p, fh, pd.partials.p, pd.rc, 1, op.slot};
      launch_boundary(op.mode, op.dot, L);
      I.note_launch("k_boundary");
    }
  CK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------
// construction
// ---------------------------------------------------------------------------------------------
Engine::Engine(Hierarchy* h, int nlocal, const int32_t* local_parts, const int32_t* device_ids, int kmax) : impl(new Impl) {
  Impl& I = *impl;
  if (kmax < 1 || kmax > PAMG_MAX_RHS) throw std::runtime_error("right-hand-side capacity must be in 1..PAMG_MAX_RHS");
  I.kmax = kmax;
  I.h = h;
  I.nparts = h->nparts;
  I.L = (int)h->levels.size();
  if (I.L > MAX_LEVELS) throw std::runtime_error("too many levels");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) throw NoGpuError("no CUDA device available (there is no CPU fallback)");
  I.local_index.assign(I.nparts, -1);
  I.arena_of.assign(I.nparts, nullptr);
  I.ipc.resize(I.nparts);
  I.have_ipc.assign(I.nparts, 0);
  const pamg_options& o = h->opts;

  // global decisions (identical in every process because the metadata is replicated)
  I.need_halo_A.assign(I.L, 0);
  I.need_halo_R.assign(I.L, 0);
  I.need_halo_P.assign(I.L, 0);
  for (int l = 0; l < I.L; ++l)
    for (int p = 0; p < I.nparts; ++p) {
      const PartLevel& pl = h->levels[l].parts[p];
      if (pl.block_nnz(PAMG_A_OG) > 0) I.need_halo_A[l] = 1;
      if (pl.block_nnz(PAMG_R_OG) > 0) I.need_halo_R[l] = 1;
      if (pl.block_nnz(PAMG_P_OG) > 0) I.need_halo_P[l] = 1;
    }

  I.tail_level = tail_level_of(*h);
  // merged (replicated) tail levels: built once on the host, uploaded to every local part's device
  std::vector<LocalCsr> tA(I.L), tP(I.L), tR(I.L);
  std::vector<std::vector<double>> tw(I.L), tdinv(I.L);
  if (I.tail_level < I.L - 1)
    for (int l = I.tail_level; l < I.L; ++l) {
      const int64_t n = h->levels[l].n_global;
      merged_block(*h, l, PAMG_A_OO, tA[l]);
      if (l + 1 < I.L) {
        merged_block(*h, l, PAMG_P_OO, tP[l]);
        merged_block(*h, l, PAMG_R_OO, tR[l]);
      }
      tw[l].assign(n, 0.0);
      tdinv[l].assign(n, 0.0);
      const double rho = h->levels[l].rho;
      const double theta = 0.5 * (o.cheb_hi_frac * rho + o.cheb_lo_frac * rho);
      for (int p = 0; p < I.nparts; ++p) {
        const PartLevel& pl = h->levels[l].parts[p];
        for (int64_t k = 0; k < pl.n_own; ++k) {
          const int64_t g = pl.own_to_global[k];
          tdinv[l][g] = 1.0 / pl.diag[k];
          if (o.smoother == PAMG_SMOOTHER_L1JACOBI)
            tw[l][g] = 1.0 / pl.diag_l1[k];
          else if (o.smoother == PAMG_SMOOTHER_CHEBYSHEV)
            tw[l][g] = (1.0 / theta) / pl.diag[k];
          else
            tw[l][g] = o.omega_jacobi / pl.diag[k];
        }
      }
    }

  for (int i = 0; i < nlocal; ++i) {
    const int part = local_parts[i];
    if (part < 0 || part >= I.nparts || I.local_index[part] >= 0) throw std::runtime_error("bad local part list");
    const int dev = device_ids ? device_ids[i] : 0;
    if (dev < 0 || dev >= ndev) throw std::runtime_error("bad device id");
    if (!h->levels[0].parts[part].full) throw std::runtime_error("local part was loaded as metadata only");
    I.local_index[part] = (int)I.parts.size();
    I.parts.emplace_back(new PartDev);
    PartDev& pd = *I.parts.back();
    pd.part = part;
    pd.device = dev;
    CK(cudaSetDevice(dev));
    if (!I.stream_of_device.count(dev)) {
      cudaStream_t s;
      CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
      I.stream_of_device[dev] = s;
    }
    pd.stream = I.stream_of_device[dev];
    CK(cudaEventCreate(&pd.ev0));
    CK(cudaEventCreate(&pd.ev1));
    pd.lay = arena_layout(*h, part);
    CK(cudaMalloc(&pd.arena, pd.lay.col_stride * kmax));
    CK(cudaMemset(pd.arena, 0, pd.lay.col_stride * kmax));
    {
      const int32_t cap = kmax;
      CK(cudaMemcpy(pd.arena + pd.lay.capacity, &cap, sizeof(cap), cudaMemcpyHostToDevice));
    }
    I.arena_of[part] = pd.arena;
    pd.cols.reset(new PartDev::Col[kmax]);
    for (int c = 0; c < kmax; ++c) {
      DBuf<DevState>& st = pd.cols[c].st;
      st.alloc(1);
      unsigned long long tmo = SPIN_TIMEOUT_NS;
      if (const char* te = getenv("PAMG_SPIN_TIMEOUT_MS")) tmo = std::max(1ll, atoll(te)) * 1000000ull;
      CK(cudaMemcpy(&st.p->spin_timeout_ns, &tmo, sizeof(tmo), cudaMemcpyHostToDevice));
    }
    pd.scratch4.alloc(RED_W);
    int max_blocks = Impl::MAX_GRID;

    for (int l = 0; l < I.L; ++l) {
      const PartLevel& pl = h->levels[l].parts[part];
      pd.lev.emplace_back(new LevelDev);
      LevelDev& ld = *pd.lev.back();
      ld.n_own = pl.n_own;
      ld.n_ghost = pl.n_ghost;
      for (int b = 0; b < 6; b += 2) {
        int lanes = 0;
        if (b == PAMG_A_OO && o.lanes_per_row > 0) lanes = o.lanes_per_row;
        build_csr(pl.blk[b], false, ld.blk[b], lanes, o.spmv_format, o, b);
        build_bnd(pl.blk[b], pl.blk[b + 1], ld.bnd[b / 2]);
        max_blocks = std::max(max_blocks, ld.blk[b].nblocks);
        max_blocks = std::max(max_blocks, (std::max(ld.blk[b].nslices, ld.blk[b].nslices4) + BLOCK / 32 - 1) / (BLOCK / 32));
      }
      // smoother weights
      std::vector<double> w(pl.n_own), dinv(pl.n_own);
      const double rho = h->levels[l].rho;
      const double lmax = o.cheb_hi_frac * rho, lmin = o.cheb_lo_frac * rho;
      const double theta = 0.5 * (lmax + lmin);
      for (int64_t k = 0; k < pl.n_own; ++k) {
        dinv[k] = 1.0 / pl.diag[k];
        if (o.smoother == PAMG_SMOOTHER_L1JACOBI)
          w[k] = 1.0 / pl.diag_l1[k];
        else if (o.smoother == PAMG_SMOOTHER_CHEBYSHEV)
          w[k] = (1.0 / theta) / pl.diag[k];
        else
          w[k] = o.omega_jacobi / pl.diag[k];
      }
      ld.w.upload(w);
      ld.dinv.upload(dinv);
      ld.send_idx.upload(pl.send_idx);
      ld.n_send = (int)pl.send_idx.size();
      ld.n_send_nbrs = (int)pl.send.size();
      ld.n_recv_nbrs = (int)pl.recv.size();
      ld.cols.reset(new LevelDev::Col[kmax]);
      for (int c = 0; c < kmax; ++c) {
        LevelDev::Col& lc = ld.cols[c];
        lc.x.alloc(pl.n_own);
        lc.x2.alloc(pl.n_own);
        lc.b.alloc(pl.n_own);
        lc.t.alloc(pl.n_own);
        if (o.smoother == PAMG_SMOOTHER_CHEBYSHEV) {
          lc.d.alloc(pl.n_own);
          lc.d2.alloc(pl.n_own);
        }
        const char* ca = pd.arena + (size_t)c * pd.lay.col_stride;
        lc.hr.ghost[0] = (const double*)(ca + pd.lay.ghost[l]);
        lc.hr.ghost[1] = lc.hr.ghost[0] + pl.n_ghost;
        lc.hr.flags = (const uint32_t*)(ca + pd.lay.flags[l]);
        lc.hr.n_nbrs = ld.n_recv_nbrs;
      }
      // assemble! gather plan: for every own row that some neighbour holds as a ghost, the staging
      // positions that contribute to it (ascending neighbour part, ascending slot).  It works on the caller's
      // local vector (io_local).
      {
        std::vector<std::vector<int32_t>> contrib(pl.n_own);
        for (size_t k = 0; k < pl.send_idx.size(); ++k) contrib[pl.send_idx[k]].push_back((int32_t)k);
        std::vector<int32_t> rows, ptr{0}, src;
        for (int64_t r = 0; r < pl.n_own; ++r)
          if (!contrib[r].empty()) {
            rows.push_back((int32_t)r);
            for (int32_t s : contrib[r]) src.push_back(s);
            ptr.push_back((int32_t)src.size());
          }
        ld.asm_nrows = (int)rows.size();
        ld.asm_rows.upload(rows);
        ld.asm_ptr.upload(ptr);
        ld.asm_src.upload(src);
        ld.asm_stage = (const double*)(pd.arena + pd.lay.asm_stage[l]);
        ld.asm_flags = (const uint32_t*)(pd.arena + pd.lay.asm_flags[l]);
      }
    }
    pd.partials_cap = max_blocks + 8 * 148;  // one partial per CTA of a fused-reduction kernel (+ halo roles)
    for (int c = 0; c < kmax; ++c) pd.cols[c].partials.alloc((size_t)pd.partials_cap);
    // replicated tail: merged levels + the maps of the level it is entered through
    pd.tlev.resize(I.L);
    if (I.tail_level < I.L - 1)
      for (int l = I.tail_level; l < I.L; ++l) {
        pd.tlev[l].reset(new LevelDev);
        LevelDev& tl = *pd.tlev[l];
        const int64_t n = h->levels[l].n_global;
        tl.n_own = n;
        tl.n_ghost = 0;
        const LocalCsr empty;
        build_csr(tA[l], false, tl.blk[PAMG_A_OO], 0, o.spmv_format, o, PAMG_A_OO);
        build_csr(tP[l], false, tl.blk[PAMG_P_OO], 0, o.spmv_format, o, PAMG_P_OO);
        build_csr(tR[l], false, tl.blk[PAMG_R_OO], 0, o.spmv_format, o, PAMG_R_OO);
        for (int b = 0; b < 3; ++b) build_bnd(empty, empty, tl.bnd[b]);
        tl.w.upload(tw[l]);
        tl.dinv.upload(tdinv[l]);
        tl.cols.reset(new LevelDev::Col[kmax]);
        for (int c = 0; c < kmax; ++c) {
          LevelDev::Col& lc = tl.cols[c];
          lc.x.alloc(n);
          lc.x2.alloc(n);
          lc.b.alloc(n);
          lc.t.alloc(n);
          if (o.smoother == PAMG_SMOOTHER_CHEBYSHEV) {
            lc.d.alloc(n);
            lc.d2.alloc(n);
          }
          lc.send_nbrs.alloc(0);
        }
        tl.send_idx.alloc(0);
      }
    const PartLevel& pc = h->levels[I.tail_level].parts[part];
    pd.inv.upload(h->coarse_inv);
    pd.own_gid_T.upload(pc.own_to_global);
    pd.ghost_gid_T.upload(pc.ghost_to_global);
    // PCG vectors on level 0
    const int64_t n0 = h->levels[0].parts[part].n_own;
    for (int c = 0; c < kmax; ++c) {
      PartDev::Col& pc = pd.cols[c];
      pc.xsol.alloc(n0);
      pc.p.alloc(n0);
      pc.q.alloc(n0);
      pc.bsave.alloc(n0);
    }
    int64_t maxloc = 0;
    for (int l = 0; l < I.L; ++l) maxloc = std::max(maxloc, h->levels[l].parts[part].n_own + h->levels[l].parts[part].n_ghost);
    pd.io_local.alloc(maxloc);
  }
  CK(cudaHostAlloc(&I.hstat_base, sizeof(HostStat) * HS_RING * kmax, cudaHostAllocMapped | cudaHostAllocPortable));
  std::memset(I.hstat_base, 0, sizeof(HostStat) * HS_RING * kmax);
  plan_buffers();
  {  // fused halo roles need every local part alone on its device (a kernel may then wait for its peers)
    std::map<int, int> per_dev;
    for (auto& up : I.parts) per_dev[up->device]++;
    bool alone = true;
    for (auto& kv : per_dev) alone = alone && kv.second == 1;
    // The double-buffered staging is race-free only if a part can never run two exchanges ahead of a part that
    // still reads its values, i.e. if on every level every part RECEIVES from exactly the parts it SENDS to
    // (DESIGN.md "Halo protocol").  Structurally symmetric operators give that; an externally uploaded or
    // non-symmetric hierarchy may not.  One stream for all parts (single-device debug layout) is ordered anyway.
    bool symmetric = true;
    for (int l = 0; l < I.L && symmetric; ++l)
      for (int p = 0; p < I.nparts && symmetric; ++p) {
        const PartLevel& pl = h->levels[l].parts[p];
        std::vector<int32_t> rs, ss;
        for (const Neighbor& nb : pl.recv) rs.push_back(nb.part);
        for (const Neighbor& nb : pl.send) ss.push_back(nb.part);
        std::sort(rs.begin(), rs.end());
        std::sort(ss.begin(), ss.end());
        if (rs != ss) symmetric = false;
      }
    const bool one_stream = per_dev.size() == 1 && nlocal == I.nparts;
    if (!symmetric && !one_stream)
      throw CommError("halo plan: a part's send-neighbour set differs from its receive-neighbour set (structurally non-symmetric "
                      "operator); the peer-memory exchange protocol needs symmetric neighbour sets on multi-GPU layouts");
    {
      const char* fe = getenv("PAMG_FOLD_CHECK");
      I.fold_check = alone && (!fe || atoi(fe) != 0);
    }
    const char* env = getenv("PAMG_FUSE_HALO");
    const bool want = env ? atoi(env) != 0 : o.fuse_halo != 0;
    I.fused_halo = want && alone && symmetric;
  }
  if (nlocal == I.nparts) connect();
}

Engine::~Engine() { delete impl; }

// decide, per level, which buffer receives the zero-guess first sweep so that the V-cycle result
// always ends in LevelDev::x whatever nu_pre / nu_post / Chebyshev degree are
void Engine::plan_buffers() {
  Impl& I = *impl;
  const pamg_options& o = I.h->opts;
  const int steps = (o.smoother == PAMG_SMOOTHER_CHEBYSHEV) ? std::max(1, o.cheb_degree) : 1;
  int flips = 1;  // prolongation writes out of place
  if (o.nu_pre > 0) flips += o.nu_pre * steps - 1;  // the zero-guess first step is written by the producer of b
  flips += o.nu_post * steps;
  auto plan = [&](LevelDev& ld) {
    for (int c = 0; c < I.kmax; ++c) ld.cols[c].xstart = (flips % 2 == 0) ? ld.cols[c].x.p : ld.cols[c].x2.p;
  };
  for (auto& up : I.parts) {
    for (auto& ld : up->lev) plan(*ld);
    for (auto& ld : up->tlev)
      if (ld) plan(*ld);
  }
  I.bind(0, true);
}

// ---------------------------------------------------------------------------------------------
// peer wiring
// ---------------------------------------------------------------------------------------------
int32_t Engine::handle_bytes() { return (int32_t)sizeof(cudaIpcMemHandle_t); }

int Engine::rhs_capacity() const { return impl->kmax; }

void Engine::export_handle(int part, void* blob) {
  Impl& I = *impl;
  if (part < 0 || part >= I.nparts || I.local_index[part] < 0) throw std::runtime_error("export: part is not local");
  PartDev& pd = I.P(I.local_index[part]);
  I.set_dev(pd);
  cudaIpcMemHandle_t hdl;
  CK(cudaIpcGetMemHandle(&hdl, pd.arena));
  std::memcpy(blob, &hdl, sizeof(hdl));
}

void Engine::import_handle(int part, const void* blob) {
  Impl& I = *impl;
  if (part < 0 || part >= I.nparts) throw std::runtime_error("import: bad part");
  if (I.local_index[part] >= 0) return;  // local parts need no handle
  std::memcpy(&I.ipc[part], blob, sizeof(cudaIpcMemHandle_t));
  I.have_ipc[part] = 1;
}

void Engine::connect() {
  Impl& I = *impl;
  if (I.connected) return;
  const Hierarchy& h = *I.h;
  if (I.parts.empty()) throw std::runtime_error("connect: no local parts");
  // same-process parts on different devices: enable peer access both ways
  for (auto& a : I.parts)
    for (auto& b : I.parts)
      if (a->device != b->device) {
        int can = 0;
        CK(cudaDeviceCanAccessPeer(&can, a->device, b->device));
        if (!can) throw CommError("devices cannot access each other's memory (P2P required)");
        CK(cudaSetDevice(a->device));
        cudaError_t e = cudaDeviceEnablePeerAccess(b->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
        cudaGetLastError();
      }
  // remote parts: map their arenas (one process per GPU => one local device)
  for (int p = 0; p < I.nparts; ++p) {
    if (I.local_index[p] >= 0) continue;
    if (!I.have_ipc[p]) throw CommError("connect: missing handle for remote part " + std::to_string(p));
    I.set_dev(I.P(0));
    void* ptr = nullptr;
    CK(cudaIpcOpenMemHandle(&ptr, I.ipc[p], cudaIpcMemLazyEnablePeerAccess));
    I.ipc_opened.push_back(ptr);
    I.arena_of[p] = (char*)ptr;
  }
  std::vector<ArenaLayout> lay(I.nparts);
  for (int p = 0; p < I.nparts; ++p) lay[p] = arena_layout(h, p);
  // every process must have allocated the same number of column copies: the wiring below addresses column c of a peer's arena
  for (int p = 0; p < I.nparts; ++p) {
    if (I.local_index[p] >= 0) continue;
    int32_t cap = 0;
    I.set_dev(I.P(0));
    CK(cudaMemcpy(&cap, I.arena_of[p] + lay[p].capacity, sizeof(cap), cudaMemcpyDeviceToHost));
    if (cap != I.kmax)
      throw CommError("connect: part " + std::to_string(p) + " was initialised with right-hand-side capacity " + std::to_string(cap) +
                      ", this process with " + std::to_string(I.kmax) + " (pamg_set_rhs_capacity must agree in every process)");
  }

  for (auto& up : I.parts)
    for (int c = 0; c < I.kmax; ++c) {
    PartDev& pd = *up;
    I.set_dev(pd);
    const int me = pd.part;
    auto arena_c = [&](int q) { return I.arena_of[q] + (size_t)c * lay[q].col_stride; };
    for (int l = 0; l < I.L; ++l) {
      const PartLevel& pl = h.levels[l].parts[me];
      LevelDev& ld = *pd.lev[l];
      std::vector<SendNbr> sn;
      std::vector<AsmSendNbr> an;
      for (const Neighbor& nb : pl.send) {
        const PartLevel& ql = h.levels[l].parts[nb.part];
        int idx = -1;
        for (size_t k = 0; k < ql.recv.size(); ++k)
          if (ql.recv[k].part == me) idx = (int)k;
        if (idx < 0) throw std::runtime_error("halo plan asymmetry");
        char* qa = arena_c(nb.part);
        SendNbr s;
        double* g0 = (double*)(qa + lay[nb.part].ghost[l]);
        s.ghost[0] = g0 + nb.slot0;
        s.ghost[1] = g0 + ql.n_ghost + nb.slot0;
        s.flag = (uint32_t*)(qa + lay[nb.part].flags[l]) + idx;
        s.offset = (int32_t)nb.offset;
        s.count = nb.count;
        sn.push_back(s);
      }
      ld.cols[c].send_nbrs.upload(sn);
      if (c > 0) continue;  // assemble! is a single-column operation
      // assemble!: my ghosts owned by q go to q's staging at the offset of q's send segment for me
      for (const Neighbor& rb : pl.recv) {
        const PartLevel& ql = h.levels[l].parts[rb.part];
        int idx = -1;
        for (size_t k = 0; k < ql.send.size(); ++k)
          if (ql.send[k].part == me) idx = (int)k;
        if (idx < 0) throw std::runtime_error("halo plan asymmetry");
        char* qa = I.arena_of[rb.part];
        AsmSendNbr a;
        a.stage[0] = (double*)(qa + lay[rb.part].asm_stage[l]) + ql.send[idx].offset;
        a.stage[1] = a.stage[0] + ql.n_send_entries();
        a.flag = (uint32_t*)(qa + lay[rb.part].asm_flags[l]) + idx;
        a.slot0 = rb.slot0;
        a.count = rb.count;
        an.push_back(a);
      }
      ld.asm_nbrs.upload(an);
    }
    std::vector<RedPub> rp(I.nparts);
    std::vector<CoarsePub> cp(I.nparts);
    for (int d = 0; d < I.nparts; ++d) {
      char* qa = arena_c(d);
      double* r0 = (double*)(qa + lay[d].red);
      rp[d].slot[0] = r0 + (size_t)me * RED_W;
      rp[d].slot[1] = r0 + (size_t)I.nparts * RED_W + (size_t)me * RED_W;
      rp[d].flag = (uint32_t*)(qa + lay[d].red_flags) + me;
      double* c0 = (double*)(qa + lay[d].coarse);
      cp[d].buf[0] = c0;
      cp[d].buf[1] = c0 + h.levels[I.tail_level].n_global;
      cp[d].flag = (uint32_t*)(qa + lay[d].coarse_flags) + me;
    }
    PartDev::Col& pc = pd.cols[c];
    pc.red_pubs.upload(rp);
    pc.coarse_pubs.upload(cp);
    pc.rc.pubs = pc.red_pubs.p;
    pc.rc.local = (const double*)(arena_c(me) + pd.lay.red);
    pc.rc.flags = (const uint32_t*)(arena_c(me) + pd.lay.red_flags);
    pc.rc.nparts = I.nparts;
  }
  I.bind(0, true);
  I.connected = true;
}

void Engine::require_connected() {
  if (!impl->connected) throw CommError("remote parts are not connected: call pamg_comm_import for every remote part, then pamg_comm_connect");
}

// ---------------------------------------------------------------------------------------------
// host <-> device vector helpers
// ---------------------------------------------------------------------------------------------
void Engine::sync_all() {
  Impl& I = *impl;
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaStreamSynchronize(up->stream));
  }
}

// host vectors: one pointer per part, column j of a multi-column call at [j * nparts + part]
void Engine::upload_vec(int level, const double* const* host, int which_buf) {
  Impl& I = *impl;
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    const double* hv = host[(size_t)I.col_of(s) * I.nparts + pd.part];
    I.set_dev(pd);
    if (!hv) throw std::runtime_error("null vector pointer for a local part");
    CK(cudaMemcpyAsync(vec(pd, level, which_buf), hv, pd.lev[level]->n_own * sizeof(double), cudaMemcpyHostToDevice, pd.stream));
  }
}

// device vector `src` of `level` (own length) -> host array (asynchronous on the part's stream)
void Engine::download_own(PartDev& pd, int level, const double* src, double* host) {
  impl->set_dev(pd);
  CK(cudaMemcpyAsync(host, src, pd.lev[level]->n_own * sizeof(double), cudaMemcpyDeviceToHost, pd.stream));
}

void Engine::download_vec(int level, double* const* host, int which_buf) {
  Impl& I = *impl;
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    double* hv = host[(size_t)I.col_of(s) * I.nparts + pd.part];
    I.set_dev(pd);
    if (!hv) throw std::runtime_error("null vector pointer for a local part");
    download_own(pd, level, vec(pd, level, which_buf), hv);
  }
  sync_all();
}

double* Engine::vec(PartDev& pd, int level, int which) {
  LevelDev& ld = *pd.lev[level];
  switch (which) {
    case V_X: return ld.x.p;
    case V_X2: return ld.x2.p;
    case V_B: return ld.b.p;
    case V_T: return ld.t.p;
    case V_XSTART: return ld.xstart;
    case V_XSOL: return pd.xsol.p;
    case V_P: return pd.p.p;
    case V_Q: return pd.q.p;
    case V_BSAVE: return pd.bsave.p;
    default: throw std::runtime_error("bad vector id");
  }
}

void Engine::check_device_error() {
  Impl& I = *impl;
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    I.set_dev(pd);
    DevState ds;
    CK(cudaMemcpy(&ds, pd.st.p, sizeof(ds), cudaMemcpyDeviceToHost));
    if (ds.error) {
      CK(cudaMemset(&pd.st.p->error, 0, sizeof(int32_t)));
      throw CommError("halo/all-reduce wait timed out on part " + std::to_string(pd.part));
    }
  }
}

void Engine::clear_done() {
  Impl& I = *impl;
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    I.set_dev(pd);
    CK(cudaMemsetAsync(&pd.st.p->done, 0, sizeof(int32_t), pd.stream));
  }
}

// ---------------------------------------------------------------------------------------------
// level operations (enqueue only)
// ---------------------------------------------------------------------------------------------
std::vector<const double*> Engine::ptrs(int level, int which) {
  std::vector<const double*> v;
  for (size_t s = 0; s < impl->nslots(); ++s) v.push_back(vec(impl->S(s), level, which));
  return v;
}

// one smoother "sweep" from `cur` into the other ping-pong buffer(s); returns the new current id.
// dot_r: fuse sum(dotv .* result) on the LAST step (level-0 post-smoothing, r.z for PCG).
void Engine::enqueue_smooth(int l, int nu, std::vector<double*>& cur, bool zero_guess_done, bool dot_last) {
  Impl& I = *impl;
  const pamg_options& o = I.h->opts;
  const size_t np = I.nslots();
  auto other = [&](size_t i) {
    LevelDev& ld = I.LV(i, l);
    return cur[i] == ld.x.p ? ld.x2.p : ld.x.p;
  };
  if (o.smoother != PAMG_SMOOTHER_CHEBYSHEV) {
    for (int s = zero_guess_done ? 1 : 0; s < nu; ++s) {
      std::vector<EpiArgs> epi(np);
      std::vector<const double*> xin(np);
      std::vector<double*> nxt(np);
      const bool dot = dot_last && s == nu - 1;
      for (size_t i = 0; i < np; ++i) {
        LevelDev& ld = I.LV(i, l);
        nxt[i] = other(i);
        xin[i] = cur[i];
        epi[i] = EpiArgs{nxt[i], ld.b.p, cur[i], ld.w.p, nullptr, nullptr, dot ? ld.b.p : nullptr, 0.0, 0.0};
      }
      OpSpec op{l, PAMG_A_OO, l, M_JACOBI, dot, 1, false};
      enqueue_op(op, xin, epi);
      cur = nxt;
    }
    return;
  }
  // Chebyshev (three-term recurrence; oracle/amg_oracle.py chebyshev())
  const double rho = I.h->levels[l].rho;
  const double lmax = o.cheb_hi_frac * rho, lmin = o.cheb_lo_frac * rho;
  const double theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin), sigma = theta / delta;
  const int deg = std::max(1, o.cheb_degree);
  for (int s = 0; s < nu; ++s) {
    double rho_k = 1.0 / sigma;
    std::vector<const double*> dcur(np, nullptr);  // d of the previous step
    for (int k = 0; k < deg; ++k) {
      const bool skip = (s == 0 && k == 0 && zero_guess_done);  // x = d = (1/theta) D^-1 b already in cur
      double c1 = 0.0, c2 = 1.0 / theta;
      if (k > 0) {
        const double rho_n = 1.0 / (2.0 * sigma - rho_k);
        c1 = rho_n * rho_k;
        c2 = 2.0 * rho_n / delta;
        rho_k = rho_n;
      }
      if (skip) {
        for (size_t i = 0; i < np; ++i) dcur[i] = cur[i];
        continue;
      }
      std::vector<EpiArgs> epi(np);
      std::vector<const double*> xin(np);
      std::vector<double*> nxt(np);
      const bool dot = dot_last && s == nu - 1 && k == deg - 1;
      for (size_t i = 0; i < np; ++i) {
        LevelDev& ld = I.LV(i, l);
        nxt[i] = other(i);
        xin[i] = cur[i];
        double* dnew = (dcur[i] == ld.d.p) ? ld.d2.p : ld.d.p;
        epi[i] = EpiArgs{nxt[i], ld.b.p, cur[i], ld.dinv.p, dnew, k > 0 ? dcur[i] : nullptr, dot ? ld.b.p : nullptr, c1, c2};
        dcur[i] = dnew;
      }
      if (dot) throw std::runtime_error("internal: fused dot is not instantiated for Chebyshev");
      OpSpec op{l, PAMG_A_OO, l, M_CHEB, false, 0, false};
      enqueue_op(op, xin, epi);
      cur = nxt;
    }
  }
}

// Levels [tail_level, L).  With only the coarsest level in the tail: all-gather b_L and apply the dense
// inverse to this part's own + ghost rows.  Otherwise: all-gather b of the first tail level, run the
// merged levels on this GPU alone (no halo), and scatter x back to this part's own + ghost slots.
void Engine::enqueue_tail(bool zero_guess) {
  Impl& I = *impl;
  const int l = I.tail_level;
  const int n = (int)I.h->levels[l].n_global;
  const pamg_options& o = I.h->opts;
  if (!zero_guess) {  // W-cycle, second visit: the right-hand side is unchanged, the merged level continues from its x
    if (l == I.L - 1) return;  // exact solve: nothing to improve
    I.tail_mode = true;
    try {
      enqueue_vcycle(l, false, false);
    } catch (...) {
      I.tail_mode = false;
      throw;
    }
    I.tail_mode = false;
    for (size_t s = 0; s < I.nslots(); ++s) {
      PartDev& pd = I.S(s);
      LevelDev& ld = *pd.lev[l];
      LevelDev& tl = *pd.tlev[l];
      I.set_dev(pd);
      k_tail_out<<<I.grid_for(std::max<int64_t>(ld.n_own + ld.n_ghost, 1), BLOCK), BLOCK, 0, pd.stream>>>(
          tl.x.p, pd.own_gid_T.p, (int)ld.n_own, pd.ghost_gid_T.p, (int)ld.n_ghost, ld.x.p, (double*)ld.hr.ghost[0], pd.st.p);
      I.note_launch("k_tail_out");
    }
    CK(cudaGetLastError());
    return;
  }
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    LevelDev& ld = *pd.lev[l];
    I.set_dev(pd);
    k_coarse_gather<<<I.grid_for(ld.n_own, BLOCK), BLOCK, 0, pd.stream>>>(ld.b.p, pd.own_gid_T.p, (int)ld.n_own, pd.coarse_pubs.p,
                                                                         I.nparts, pd.st.p);
    I.note_launch("k_coarse_gather");
  }
  if (l == I.L - 1) {
    for (size_t s = 0; s < I.nslots(); ++s) {
      PartDev& pd = I.S(s);
      LevelDev& ld = *pd.lev[l];
      I.set_dev(pd);
      const int rows = (int)(ld.n_own + ld.n_ghost);
      const double* c0 = (const double*)(pd.carena + pd.lay.coarse);
      k_coarse_solve<<<I.grid_for(std::max(rows, 1), BLOCK / 32), BLOCK, 0, pd.stream>>>(
          pd.inv.p, n, c0, c0 + n, (const uint32_t*)(pd.carena + pd.lay.coarse_flags), I.nparts, pd.own_gid_T.p, (int)ld.n_own,
          pd.ghost_gid_T.p, (int)ld.n_ghost, ld.x.p, (double*)ld.hr.ghost[0], pd.st.p);
      I.note_launch("k_coarse_solve");
    }
    CK(cudaGetLastError());
    return;
  }
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    LevelDev& tl = *pd.tlev[l];
    I.set_dev(pd);
    const double* c0 = (const double*)(pd.carena + pd.lay.coarse);
    k_tail_in<<<I.grid_for(n, BLOCK), BLOCK, 0, pd.stream>>>(c0, c0 + n, (const uint32_t*)(pd.carena + pd.lay.coarse_flags), I.nparts,
                                                             tl.b.p, tl.xstart, o.nu_pre > 0 ? tl.w.p : nullptr, n, pd.st.p);
    I.note_launch("k_tail_in");
  }
  CK(cudaGetLastError());
  I.tail_mode = true;
  try {
    enqueue_vcycle(l, false, true);
  } catch (...) {
    I.tail_mode = false;
    throw;
  }
  I.tail_mode = false;
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    LevelDev& ld = *pd.lev[l];
    LevelDev& tl = *pd.tlev[l];
    I.set_dev(pd);
    k_tail_out<<<I.grid_for(std::max<int64_t>(ld.n_own + ld.n_ghost, 1), BLOCK), BLOCK, 0, pd.stream>>>(
        tl.x.p, pd.own_gid_T.p, (int)ld.n_own, pd.ghost_gid_T.p, (int)ld.n_ghost, ld.x.p, (double*)ld.hr.ghost[0], pd.st.p);
    I.note_launch("k_tail_out");
  }
  CK(cudaGetLastError());
}

// V-cycle from level l.  Preconditions: lev[l].b holds the right-hand side and lev[l].xstart holds
// the zero-guess first pre-smoothing step (w .* b, or 0 when nu_pre == 0).  Result in lev[l].x.
// zero_guess == false (W-cycle, second visit of a level): continue from the current lev[l].x with full pre-smoothing.
void Engine::enqueue_vcycle(int l, bool dot_rz, bool zero_guess) {
  Impl& I = *impl;
  const pamg_options& o = I.h->opts;
  const size_t np = I.nslots();
  if (!I.tail_mode && l == I.tail_level) {
    enqueue_tail(zero_guess);
    return;
  }
  if (I.tail_mode && l == I.L - 1) {  // coarsest level of the replicated tail: x = A_L^-1 b, whole vector
    for (size_t s = 0; s < I.nslots(); ++s) {
      PartDev& pd = I.S(s);
      LevelDev& ld = I.LV(pd, l);
      I.set_dev(pd);
      k_dense<<<I.grid_for(std::max<int64_t>(ld.n_own, 1), BLOCK / 32), BLOCK, 0, pd.stream>>>(pd.inv.p, (int)ld.n_own, ld.b.p, ld.x.p,
                                                                                             pd.st.p);
      I.note_launch("k_dense");
    }
    CK(cudaGetLastError());
    return;
  }
  // the next level is entered through the tail gather / the dense solve: no fused zero-guess step for it
  const bool next_is_entry = I.tail_mode ? (l + 1 == I.L - 1) : (l + 1 == I.tail_level);
  std::vector<double*> cur(np);
  for (size_t i = 0; i < np; ++i) cur[i] = zero_guess ? I.LV(i, l).xstart : I.LV(i, l).x.p;
  if (o.nu_pre > 0) enqueue_smooth(l, o.nu_pre, cur, /*zero_guess_done=*/zero_guess, false);
  // residual t = b - A x
  {
    std::vector<EpiArgs> epi(np);
    std::vector<const double*> xin(np);
    for (size_t i = 0; i < np; ++i) {
      LevelDev& ld = I.LV(i, l);
      xin[i] = cur[i];
      epi[i] = EpiArgs{ld.t.p, ld.b.p, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
    }
    OpSpec op{l, PAMG_A_OO, l, M_RESID, false, 0, false};
    enqueue_op(op, xin, epi);
  }
  // restriction b_c = R t, fused with the coarse level's zero-guess first smoothing step
  {
    const bool coarse_is_last = next_is_entry;
    std::vector<EpiArgs> epi(np);
    std::vector<const double*> xin(np);
    for (size_t i = 0; i < np; ++i) {
      LevelDev& ld = I.LV(i, l);
      LevelDev& lc = I.LV(i, l + 1);
      xin[i] = ld.t.p;
      double* out2 = coarse_is_last ? nullptr : lc.xstart;
      const double* w = (o.nu_pre > 0) ? lc.w.p : nullptr;
      epi[i] = EpiArgs{lc.b.p, nullptr, nullptr, w, out2, nullptr, nullptr, 0.0, 0.0};
      if (out2 && !w) epi[i].out2 = nullptr;  // nu_pre == 0: xstart is zeroed below instead
    }
    OpSpec op{l, PAMG_R_OO, l, M_RESTRICT, false, 0, false};
    enqueue_op(op, xin, epi);
    if (!coarse_is_last && o.nu_pre == 0)
      for (size_t i = 0; i < np; ++i) {
        PartDev& pd = I.S(i);
        LevelDev& lc = I.LV(pd, l + 1);
        I.set_dev(pd);
        k_scale<<<I.grid_for(lc.n_own, BLOCK * 4), BLOCK, 0, pd.stream>>>(lc.b.p, nullptr, lc.xstart, (int)lc.n_own, pd.st.p);
        I.note_launch("k_scale");
      }
  }
  enqueue_vcycle(l + 1, false, true);
  // W-cycle: the coarse problem is visited a second time, from the first visit's result (the coarsest solve is exact)
  if (o.cycle == PAMG_CYCLE_W && l + 1 < I.L - 1) enqueue_vcycle(l + 1, false, false);
  // prolongation + correction (out of place): nxt = cur + P e_c
  {
    std::vector<EpiArgs> epi(np);
    std::vector<const double*> xin(np);
    std::vector<double*> nxt(np);
    for (size_t i = 0; i < np; ++i) {
      LevelDev& ld = I.LV(i, l);
      LevelDev& lc = I.LV(i, l + 1);
      nxt[i] = (cur[i] == ld.x.p) ? ld.x2.p : ld.x.p;
      xin[i] = lc.x.p;
      epi[i] = EpiArgs{nxt[i], cur[i], nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
    }
    OpSpec op{l, PAMG_P_OO, l + 1, M_ADD, false, 0, !I.tail_mode && l + 1 == I.tail_level};
    enqueue_op(op, xin, epi);
    cur = nxt;
  }
  if (o.nu_post > 0) enqueue_smooth(l, o.nu_post, cur, false, dot_rz);
  for (size_t i = 0; i < np; ++i) {
    LevelDev& ld = I.LV(i, l);
    if (cur[i] == ld.x.p) continue;
    if (zero_guess) throw std::runtime_error("internal: V-cycle buffer plan mismatch");
    // a visit that started from x has one buffer flip more than the plan of the zero-guess visit: copy back
    PartDev& pd = I.S(i);
    I.set_dev(pd);
    k_copy<<<I.grid_for(ld.n_own, BLOCK * 4), BLOCK, 0, pd.stream>>>(cur[i], ld.x.p, (int)ld.n_own, pd.st.p);
    I.note_launch("k_copy");
  }
}

// r.z when the V-cycle could not fuse it (nu_post == 0, Chebyshev, or a single-level hierarchy)
void Engine::enqueue_dot_rz() {
  Impl& I = *impl;
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    LevelDev& l0 = *pd.lev[0];
    I.set_dev(pd);
    k_dot<<<I.grid_red(l0.n_own), BLOCK, 0, pd.stream>>>(l0.b.p, l0.x.p, (int)l0.n_own, pd.st.p, pd.partials.p, pd.rc,
                                                                   1, 1);
    I.note_launch("k_dot");
  }
  CK(cudaGetLastError());
}

bool Engine::vcycle_fuses_rz() const {
  const pamg_options& o = impl->h->opts;
  return impl->L > 1 && o.nu_post > 0 && o.smoother != PAMG_SMOOTHER_CHEBYSHEV;
}

// one PCG iteration (uniform body, see DESIGN.md "PCG schedule"):
//   z = M^-1 r (rz fused) ; beta = rz/rho_old ; p = z + beta p ; q = A p (pq fused) ;
//   alpha = rz/pq ; x += alpha p ; r -= alpha q ; z0 = w .* r ; rr ; check
void Engine::enqueue_pcg_iteration(int mode) {
  Impl& I = *impl;
  const size_t np = I.nslots();
  const bool precond = mode != 0, flexible = mode == 2;
  if (flexible) {  // z = M^-1 r, then r.z and r_prev.z in one pass (one all-reduce)
    enqueue_vcycle(0, false, true);
    for (size_t s = 0; s < I.nslots(); ++s) {
      PartDev& pd = I.S(s);
      LevelDev& l0 = *pd.lev[0];
      I.set_dev(pd);
      k_dot2<<<I.grid_red(l0.n_own), BLOCK, 0, pd.stream>>>(l0.b.p, l0.x.p, pd.rprev.p, (int)l0.n_own, pd.st.p, pd.partials.p, pd.rc);
      I.note_launch("k_dot2");
    }
  } else if (precond) {
    enqueue_vcycle(0, vcycle_fuses_rz(), true);
    if (!vcycle_fuses_rz()) enqueue_dot_rz();
  } else {
    for (size_t s = 0; s < I.nslots(); ++s) {
      PartDev& pd = I.S(s);
      LevelDev& l0 = *pd.lev[0];
      I.set_dev(pd);
      k_copy_dot<<<I.grid_red(l0.n_own), BLOCK, 0, pd.stream>>>(l0.b.p, l0.x.p, (int)l0.n_own, pd.st.p, pd.partials.p,
                                                                          pd.rc);
      I.note_launch("k_copy_dot");
    }
  }
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    LevelDev& l0 = *pd.lev[0];
    I.set_dev(pd);
    k_update_p<<<I.grid_for(l0.n_own, BLOCK * 4), BLOCK, 0, pd.stream>>>(l0.x.p, pd.p.p, (int)l0.n_own, pd.st.p, pd.rc, flexible ? 1 : 0);
    I.note_launch("k_update_p");
  }
  {
    std::vector<EpiArgs> epi(np);
    std::vector<const double*> xin(np);
    for (size_t i = 0; i < np; ++i) {
      PartDev& pd = I.S(i);
      xin[i] = pd.p.p;
      epi[i] = EpiArgs{pd.q.p, nullptr, nullptr, nullptr, nullptr, nullptr, pd.p.p, 0.0, 0.0};
    }
    OpSpec op{0, PAMG_A_OO, 0, M_MUL, true, 2, false};
    enqueue_op(op, xin, epi);
  }
  const bool zero_guess = precond && I.L > 1 && I.h->opts.nu_pre > 0;
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    LevelDev& l0 = *pd.lev[0];
    I.set_dev(pd);
    k_update_xr<<<I.grid_red(l0.n_own), BLOCK, 0, pd.stream>>>(pd.xsol.p, l0.b.p, pd.p.p, pd.q.p, l0.xstart,
                                                                         zero_guess ? l0.w.p : nullptr, (int)l0.n_own, pd.st.p,
                                                                         pd.partials.p, pd.rc, I.fold_check ? 1 : 0, pd.hist.p,
                                                                         &pd == I.parts[0].get() ? I.hstat : nullptr,
                                                                         flexible ? pd.rprev.p : nullptr);
    I.note_launch(I.fold_check ? "k_update_xr+check" : "k_update_xr");
  }
  if (!I.fold_check)  // several parts on one GPU: a kernel must not wait for a later kernel of its own stream
    for (size_t s = 0; s < I.nslots(); ++s) {
      PartDev& pd = I.S(s);
      I.set_dev(pd);
      k_check<<<1, 1, 0, pd.stream>>>(pd.st.p, pd.rc, pd.hist.p, &pd == I.parts[0].get() ? I.hstat : nullptr);
      I.note_launch("k_check");
    }
  CK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------
// graph capture over all local streams
// ---------------------------------------------------------------------------------------------
template <class F>
void Engine::capture(std::vector<cudaGraphExec_t>& out, int64_t* nodes, F&& body) {
  Impl& I = *impl;
  for (auto g : out) cudaGraphExecDestroy(g);
  out.clear();
  I.g_streams.clear();
  for (auto& kv : I.stream_of_device) I.g_streams.push_back(kv.second);
  std::vector<int> devs;
  for (auto& kv : I.stream_of_device) devs.push_back(kv.first);
  for (size_t k = 0; k < I.g_streams.size(); ++k) {
    CK(cudaSetDevice(devs[k]));
    CK(cudaStreamBeginCapture(I.g_streams[k], cudaStreamCaptureModeRelaxed));
  }
  const int64_t before = I.launches;
  std::string err;
  try {
    body();
  } catch (const std::exception& e) {
    err = e.what();
  }
  *nodes = I.launches - before;
  I.launches = before;
  for (size_t k = 0; k < I.g_streams.size(); ++k) {
    CK(cudaSetDevice(devs[k]));
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(I.g_streams[k], &g);
    if (e != cudaSuccess && err.empty()) err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e);
    if (g && err.empty()) {
      cudaGraphExec_t ge = nullptr;
      e = cudaGraphInstantiate(&ge, g, 0);
      if (e != cudaSuccess)
        err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e);
      else
        out.push_back(ge);
    }
    if (g) cudaGraphDestroy(g);
  }
  if (!err.empty()) throw CudaError("graph capture failed: " + err);
}

void Engine::launch_graphs(const std::vector<cudaGraphExec_t>& gs, int64_t nodes) {
  Impl& I = *impl;
  size_t k = 0;
  for (auto& kv : I.stream_of_device) {
    CK(cudaSetDevice(kv.first));
    CK(cudaGraphLaunch(gs[k], kv.second));
    ++k;
  }
  I.launches += nodes;
}

// ---------------------------------------------------------------------------------------------
// public operations
// ---------------------------------------------------------------------------------------------
void Engine::spmv(int level, const double* const* x, double* const* y) {
  require_connected();
  Impl& I = *impl;
  if (level < 0 || level >= I.L) throw std::runtime_error("bad level");
  I.launches = 0;
  clear_done();
  upload_vec(level, x, V_X);
  const size_t ns = I.nslots();
  std::vector<EpiArgs> epi(ns);
  for (size_t s = 0; s < ns; ++s)
    epi[s] = EpiArgs{I.S(s).lev[level]->t.p, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
  OpSpec op{level, PAMG_A_OO, level, M_MUL, false, 0, false};
  enqueue_op(op, ptrs(level, V_X), epi);
  download_vec(level, y, V_T);
  check_device_error();
}

void Engine::smooth(int level, int nu, const double* const* b, double* const* x) {
  require_connected();
  Impl& I = *impl;
  if (level < 0 || level >= I.L) throw std::runtime_error("bad level");
  I.launches = 0;
  clear_done();
  upload_vec(level, b, V_B);
  upload_vec(level, x, V_X);
  std::vector<double*> cur;
  for (auto& up : I.parts) cur.push_back(up->lev[level]->x.p);
  enqueue_smooth(level, nu, cur, false, false);
  for (size_t i = 0; i < I.parts.size(); ++i) {
    PartDev& pd = I.P(i);
    I.set_dev(pd);
    download_own(pd, level, cur[i], x[pd.part]);
  }
  sync_all();
  check_device_error();
}

void Engine::residual_restrict(int level, const double* const* b, const double* const* x, double* const* r, double* const* bc) {
  require_connected();
  Impl& I = *impl;
  if (level < 0 || level >= I.L - 1) throw std::runtime_error("bad level");
  I.launches = 0;
  clear_done();
  upload_vec(level, b, V_B);
  upload_vec(level, x, V_X);
  const size_t np = I.parts.size();
  std::vector<EpiArgs> epi(np);
  for (size_t i = 0; i < np; ++i) {
    LevelDev& ld = *I.P(i).lev[level];
    epi[i] = EpiArgs{ld.t.p, ld.b.p, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
  }
  OpSpec op{level, PAMG_A_OO, level, M_RESID, false, 0, false};
  enqueue_op(op, ptrs(level, V_X), epi);
  for (size_t i = 0; i < np; ++i) {
    LevelDev& lc = *I.P(i).lev[level + 1];
    epi[i] = EpiArgs{lc.b.p, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
  }
  OpSpec op2{level, PAMG_R_OO, level, M_RESTRICT, false, 0, false};
  enqueue_op(op2, ptrs(level, V_T), epi);
  if (r) download_vec(level, r, V_T);
  download_vec(level + 1, bc, V_B);
  check_device_error();
}

void Engine::prolong_correct(int level, const double* const* ec, double* const* x) {
  require_connected();
  Impl& I = *impl;
  if (level < 0 || level >= I.L - 1) throw std::runtime_error("bad level");
  I.launches = 0;
  clear_done();
  upload_vec(level, x, V_X);
  upload_vec(level + 1, ec, V_X);
  const size_t np = I.parts.size();
  std::vector<EpiArgs> epi(np);
  for (size_t i = 0; i < np; ++i) {
    LevelDev& ld = *I.P(i).lev[level];
    epi[i] = EpiArgs{ld.x2.p, ld.x.p, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
  }
  OpSpec op{level, PAMG_P_OO, level + 1, M_ADD, false, 0, false};
  enqueue_op(op, ptrs(level + 1, V_X), epi);
  download_vec(level, x, V_X2);
  check_device_error();
}

double Engine::dot(int level, const double* const* u, const double* const* v) {
  require_connected();
  Impl& I = *impl;
  if (level < 0 || level >= I.L) throw std::runtime_error("bad level");
  I.launches = 0;
  upload_vec(level, u, V_X);
  upload_vec(level, v, V_B);
  for (auto& up : I.parts) {
    PartDev& pd = *up;
    LevelDev& ld = *pd.lev[level];
    I.set_dev(pd);
    k_dot<<<I.grid_red(ld.n_own), BLOCK, 0, pd.stream>>>(ld.x.p, ld.b.p, (int)ld.n_own, pd.st.p, pd.partials.p, pd.rc, 3, 0);
    I.note_launch("k_dot");
  }
  double out[RED_W] = {0, 0, 0, 0};
  for (auto& up : I.parts) {
    PartDev& pd = *up;
    I.set_dev(pd);
    k_red_read<<<1, 1, 0, pd.stream>>>(pd.st.p, pd.rc, pd.scratch4.p);
    I.note_launch("k_red_read");
  }
  CK(cudaGetLastError());
  sync_all();
  I.set_dev(I.P(0));
  CK(cudaMemcpy(out, I.P(0).scratch4.p, sizeof(out), cudaMemcpyDeviceToHost));
  check_device_error();
  return out[3];
}

void Engine::consistent(int level, double* const* v) {
  require_connected();
  Impl& I = *impl;
  if (level < 0 || level >= I.L) throw std::runtime_error("bad level");
  I.launches = 0;
  clear_done();
  upload_vec(level, v, V_X);
  for (auto& up : I.parts) {
    PartDev& pd = *up;
    LevelDev& ld = *pd.lev[level];
    if (ld.n_send_nbrs == 0 && ld.n_recv_nbrs == 0) continue;
    I.set_dev(pd);
    k_halo_pack<<<I.grid_for(ld.n_send, BLOCK * 4), BLOCK, 0, pd.stream>>>(ld.x.p, ld.send_idx.p, ld.n_send, ld.send_nbrs.p,
                                                                           ld.n_send_nbrs, pd.st.p, level);
    I.note_launch("k_halo_pack");
  }
  for (auto& up : I.parts) {
    PartDev& pd = *up;
    LevelDev& ld = *pd.lev[level];
    if (ld.n_recv_nbrs == 0) continue;
    I.set_dev(pd);
    k_halo_unpack<<<I.grid_for(ld.n_ghost, BLOCK * 4), BLOCK, 0, pd.stream>>>(pd.io_local.p, ld.hr, (int)ld.n_ghost, pd.st.p, level);
    I.note_launch("k_halo_unpack");
    CK(cudaMemcpyAsync(v[pd.part] + ld.n_own, pd.io_local.p, ld.n_ghost * sizeof(double), cudaMemcpyDeviceToHost, pd.stream));
  }
  CK(cudaGetLastError());
  sync_all();
  check_device_error();
}

void Engine::assemble(int level, double* const* v) {
  require_connected();
  Impl& I = *impl;
  if (level < 0 || level >= I.L) throw std::runtime_error("bad level");
  I.launches = 0;
  for (auto& up : I.parts) {
    PartDev& pd = *up;
    LevelDev& ld = *pd.lev[level];
    I.set_dev(pd);
    CK(cudaMemcpyAsync(pd.io_local.p, v[pd.part], (ld.n_own + ld.n_ghost) * sizeof(double), cudaMemcpyHostToDevice, pd.stream));
    if (ld.n_send_nbrs == 0 && ld.n_recv_nbrs == 0) continue;
    k_asm_pack<<<I.grid_for(ld.n_ghost, BLOCK * 4), BLOCK, 0, pd.stream>>>(pd.io_local.p + ld.n_own, ld.asm_nbrs.p, ld.n_recv_nbrs,
                                                                           pd.st.p, level);
    I.note_launch("k_asm_pack");
  }
  for (auto& up : I.parts) {
    PartDev& pd = *up;
    LevelDev& ld = *pd.lev[level];
    I.set_dev(pd);
    if (ld.n_send_nbrs > 0) {
      k_asm_add<<<I.grid_for(std::max(ld.asm_nrows, 1), BLOCK), BLOCK, 0, pd.stream>>>(
          pd.io_local.p, ld.asm_rows.p, ld.asm_ptr.p, ld.asm_src.p, ld.asm_nrows, ld.asm_stage, ld.asm_stage + ld.n_send, ld.asm_flags,
          ld.n_send_nbrs,
          pd.st.p, level);
      I.note_launch("k_asm_add");
    }
    CK(cudaMemsetAsync(pd.io_local.p + ld.n_own, 0, ld.n_ghost * sizeof(double), pd.stream));
    CK(cudaMemcpyAsync(v[pd.part], pd.io_local.p, (ld.n_own + ld.n_ghost) * sizeof(double), cudaMemcpyDeviceToHost, pd.stream));
  }
  CK(cudaGetLastError());
  sync_all();
  check_device_error();
}

void Engine::enqueue_vcycle_entry() {
  // b is in lev[0].b; write the zero-guess first step into xstart, then the cycle
  Impl& I = *impl;
  const pamg_options& o = I.h->opts;
  if (I.L > 1)
    for (size_t s = 0; s < I.nslots(); ++s) {
      PartDev& pd = I.S(s);
      LevelDev& l0 = *pd.lev[0];
      I.set_dev(pd);
      k_scale<<<I.grid_for(l0.n_own, BLOCK * 4), BLOCK, 0, pd.stream>>>(l0.b.p, o.nu_pre > 0 ? l0.w.p : nullptr, l0.xstart,
                                                                       (int)l0.n_own, pd.st.p);
      I.note_launch("k_scale");
    }
  enqueue_vcycle(0, false, true);
}

void Engine::vcycle(const double* const* b, double* const* x) {
  require_connected();
  Impl& I = *impl;
  I.launches = 0;
  clear_done();
  upload_vec(0, b, V_B);
  const bool use_graph = I.h->opts.use_graph != 0;
  // multi-column cycles have a graph of their own, captured for the last column count
  std::vector<cudaGraphExec_t>& graph = I.multi ? I.g_vcycle_multi : I.g_vcycle;
  int64_t& nodes = I.multi ? I.g_vcycle_multi_nodes : I.g_vcycle_nodes;
  if (I.multi && I.g_vcycle_multi_k != (int)I.cols.size()) {
    for (auto g : graph) cudaGraphExecDestroy(g);
    graph.clear();
  }
  if (use_graph && graph.empty()) {
    capture(graph, &nodes, [&] { enqueue_vcycle_entry(); });
    if (I.multi) I.g_vcycle_multi_k = (int)I.cols.size();
  }
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaEventRecord(up->ev0, up->stream));
  }
  if (use_graph)
    launch_graphs(graph, nodes);
  else
    enqueue_vcycle_entry();
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaEventRecord(up->ev1, up->stream));
  }
  download_vec(0, x, V_X);
  float ms = 0, mx = 0;
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaEventElapsedTime(&ms, up->ev0, up->ev1));
    mx = std::max(mx, ms);
  }
  I.stats.vcycle_ms = mx;
  I.stats.kernel_launches = I.launches;
  check_device_error();
}

void Engine::load_rhs(const double* const* b) {
  upload_vec(0, b, V_BSAVE);
  sync_all();
  impl->rhs_loaded = true;
}

void Engine::read_solution(double* const* x) { download_vec(0, x, V_XSOL); }

int Engine::pcg(const double* const* b, double* const* x, double rtol, int maxiter, int mode, int* iters, double* hist) {
  load_rhs(b);
  int rc = pcg_resident(rtol, maxiter, mode, iters, hist);
  read_solution(x);
  return rc;
}

int Engine::pcg_resident(double rtol, int maxiter, int mode, int* iters, double* hist) {
  require_connected();
  if (!impl->rhs_loaded) throw std::runtime_error("pamg_pcg_resident: call pamg_load_rhs first");
  return run_pcg(rtol, maxiter, mode, iters, nullptr, hist);
}

// mode: 0 plain CG, 1 AMG-preconditioned CG, 2 flexible AMG-preconditioned CG.  Runs the columns I.cols (right-hand sides in
// bsave), each with its own scalars, history and convergence decision; iters / converged / hist (rows of maxiter + 1) per column.
int Engine::run_pcg(double rtol, int maxiter, int mode, int* iters, int* converged, double* hist) {
  Impl& I = *impl;
  if (maxiter < 0) throw std::runtime_error("maxiter < 0");
  if (mode < 0 || mode > 2) throw std::runtime_error("bad Krylov mode");
  const bool precond = mode != 0;
  const int graph_k = I.multi ? (int)I.cols.size() : 0;
  auto drop_graph = [&] {
    for (auto g : I.g_iter) cudaGraphExecDestroy(g);
    I.g_iter.clear();
  };
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    PartDev::Col& pc = pd.cols[I.col_of(s)];
    I.set_dev(pd);
    if (mode == 2 && pc.rprev.n == 0) {
      pc.rprev.alloc((size_t)pd.lev[0]->n_own);
      drop_graph();
    }
    if (pc.hist_cap < maxiter + 2) {
      pc.hist.alloc(maxiter + 2);
      pc.hist_cap = maxiter + 2;
      drop_graph();  // hist pointer is baked into the graph
    }
    I.bind(I.col_of(s), true);
  }
  I.launches = 0;
  const bool use_graph = I.h->opts.use_graph != 0;
  if (use_graph && (I.g_iter.empty() || I.g_iter_mode != mode || I.g_iter_k != graph_k)) {
    I.names.clear();
    I.naming = true;
    try {
      capture(I.g_iter, &I.g_iter_nodes, [&] { enqueue_pcg_iteration(mode); });
    } catch (...) {
      I.naming = false;
      throw;
    }
    I.naming = false;
    I.g_iter_mode = mode;
    I.g_iter_k = graph_k;
  }
  const bool zero_guess = precond && I.L > 1 && I.h->opts.nu_pre > 0;
  sync_all();
  for (int c : I.cols) std::memset(I.hstat_base + (size_t)c * HS_RING, 0, sizeof(HostStat) * HS_RING);
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaEventRecord(up->ev0, up->stream));
  }
  for (size_t s = 0; s < I.nslots(); ++s) {
    PartDev& pd = I.S(s);
    LevelDev& l0 = *pd.lev[0];
    I.set_dev(pd);
    k_pcg_init<<<I.grid_red(l0.n_own), BLOCK, 0, pd.stream>>>(pd.bsave.p, pd.xsol.p, l0.b.p, pd.p.p, l0.xstart,
                                                                        zero_guess ? l0.w.p : nullptr, (int)l0.n_own, pd.st.p,
                                                                        pd.partials.p, pd.rc, rtol, maxiter, I.fold_check ? 1 : 0,
                                                                        pd.hist.p, &pd == I.parts[0].get() ? I.hstat : nullptr);
    I.note_launch("k_pcg_init");
  }
  if (!I.fold_check)
    for (size_t s = 0; s < I.nslots(); ++s) {
      PartDev& pd = I.S(s);
      I.set_dev(pd);
      k_check<<<1, 1, 0, pd.stream>>>(pd.st.p, pd.rc, pd.hist.p, &pd == I.parts[0].get() ? I.hstat : nullptr);
      I.note_launch("k_check");
    }
  CK(cudaGetLastError());
  // speculative enqueue: iteration k+1 is launched before the status of iteration k is known; every
  // kernel early-outs once the device-side `done` flag is set, so the extra launch is a no-op.
  PartDev& p0 = I.P(0);
  const int LOOKAHEAD = 1;
  if (maxiter + 2 >= (1 << 30)) throw std::runtime_error("maxiter too large");
  const size_t nc = I.cols.size();
  std::vector<char> col_done(nc, 0);  // a column that reported done or error is frozen: its ring is not waited for again
  bool finished = false;
  int launched = 0;
  while (!finished) {
    if (launched < maxiter) {
      if (use_graph) {
        launch_graphs(I.g_iter, I.g_iter_nodes);
      } else {
        if (launched == 0) {
          I.names.clear();
          I.naming = true;
        }
        enqueue_pcg_iteration(mode);
        I.naming = false;
      }
    }
    ++launched;
    if (launched > LOOKAHEAD) {  // status written by k_check number (launched - LOOKAHEAD + 1), straight into pinned memory
      // k_check number 1 is the one of r0, number k + 1 the one of iteration k; none exists beyond maxiter + 1
      const uint32_t want = (uint32_t)std::min(launched - LOOKAHEAD + 1, maxiter + 1);
      bool all = true;
      for (size_t c = 0; c < nc; ++c) {
        if (col_done[c]) continue;
        volatile HostStat* hsl = I.hstat_base + (size_t)I.cols[c] * HS_RING + (want % HS_RING);
        const auto t0 = std::chrono::steady_clock::now();
        while (hsl->seq != want) {
          if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(30))
            throw CommError("timed out waiting for the device status of a PCG iteration");
        }
        if (hsl->done || hsl->error) col_done[c] = 1;
        all = all && col_done[c];
      }
      if (all) finished = true;
    }
    if (launched > maxiter + LOOKAHEAD + 1) finished = true;
  }
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaEventRecord(up->ev1, up->stream));
  }
  sync_all();
  float ms = 0, mx = 0;
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaEventElapsedTime(&ms, up->ev0, up->ev1));
    mx = std::max(mx, ms);
  }
  check_device_error();
  bool all_conv = true;
  int max_iters = 0;
  for (size_t c = 0; c < nc; ++c) {
    DevState fin;
    I.bind(I.cols[c]);
    I.set_dev(p0);
    CK(cudaMemcpy(&fin, p0.st.p, sizeof(fin), cudaMemcpyDeviceToHost));
    const double r0 = std::sqrt(fin.sc[SC_RR0]), rn = std::sqrt(fin.sc[SC_RR]);
    const bool conv = rn <= rtol * r0;
    if (iters) iters[c] = fin.iters;
    if (converged) converged[c] = conv ? 1 : 0;
    if (hist && fin.iters >= 0)
      CK(cudaMemcpy(hist + c * (size_t)(maxiter + 1), p0.hist.p, (fin.iters + 1) * sizeof(double), cudaMemcpyDeviceToHost));
    all_conv = all_conv && conv;
    max_iters = std::max(max_iters, (int)fin.iters);
    if (c == 0) {
      I.stats.r0_norm = r0;
      I.stats.r_norm = rn;
    }
  }
  I.stats.iters = max_iters;
  I.stats.converged = all_conv;
  I.stats.solve_ms = mx;
  I.stats.kernel_launches = I.launches;
  return all_conv ? PAMG_OK : PAMG_ERR_NOTCONV;
}

// ---------------------------------------------------------------------------------------------
// several right-hand sides (columns 0..k-1 of the per-solve state): the enqueue_* functions run over all of them, with k-wide
// launches where the block's kernel has one (enqueue_op) and the single-column kernels per column elsewhere
// ---------------------------------------------------------------------------------------------
void Engine::begin_multi(int k) {
  Impl& I = *impl;
  if (k < 1 || k > I.kmax)
    throw std::runtime_error("k = " + std::to_string(k) + " right-hand sides exceed the capacity " + std::to_string(I.kmax) +
                             " this device state was initialised with (pamg_set_rhs_capacity before pamg_device_init)");
  require_connected();
  I.cols.resize(k);
  for (int c = 0; c < k; ++c) I.cols[c] = c;
  I.multi = true;
}

void Engine::end_multi() {
  Impl& I = *impl;
  I.cols.assign(1, 0);
  I.multi = false;
  I.bind(0);
}

template <class F>
auto Engine::in_multi(int k, F&& body) -> decltype(body()) {
  begin_multi(k);
  try {
    auto r = body();
    end_multi();
    return r;
  } catch (...) {
    end_multi();
    throw;
  }
}

// kernel timing of k columns (kinds whose operations run through enqueue_op: 0, 1, 2, 3, 6, 7), so a k-wide launch can be
// compared with k single launches of the same block (scripts/multi_rhs_sweep.py)
void Engine::time_kernel_multi(int k, int kind, int level, int reps, bool flush_l2, float* ms_out) {
  if (kind != 0 && kind != 1 && kind != 2 && kind != 3 && kind != 6 && kind != 7)
    throw std::runtime_error("multi-column timing covers kinds 0, 1, 2, 3, 6 and 7");
  in_multi(k, [&] {
    time_kernel(kind, level, reps, flush_l2, ms_out);
    return 0;
  });
}

void Engine::spmv_multi(int level, int k, const double* const* x, double* const* y) {
  in_multi(k, [&] {
    spmv(level, x, y);
    return 0;
  });
}

void Engine::vcycle_multi(int k, const double* const* b, double* const* x) {
  in_multi(k, [&] {
    vcycle(b, x);
    return 0;
  });
}

int Engine::pcg_multi(int k, const double* const* b, double* const* x, double rtol, int maxiter, int mode, int* iters, int* converged,
                      double* hist) {
  return in_multi(k, [&] {
    load_rhs(b);
    const int rc = run_pcg(rtol, maxiter, mode, iters, converged, hist);
    read_solution(x);
    return rc;
  });
}

// ---------------------------------------------------------------------------------------------
// restarted flexible GMRES (oracle/amg_oracle.py fgmres, pamg_oracle.c orc_fgmres)
// ---------------------------------------------------------------------------------------------
// Host-driven: the cycle (one graph replay), the SpMV (fused halo roles as in PCG) and the modified Gram-Schmidt chain
// (k_dot -> k_gs_sub pairs: the coefficient goes from the all-reduce straight into the update) are enqueued per inner
// step; one Hessenberg column comes back per step for the Givens rotations, the residual estimate and the stopping
// decision.  Every part reads bit-identical all-reduce results, so every rank of a one-process-per-GPU job takes the
// same decisions without talking to the others.
int Engine::fgmres(const double* const* b, double* const* x, double rtol, int maxiter, int restart, int precond, int* iters,
                   double* hist) {
  require_connected();
  Impl& I = *impl;
  if (maxiter < 0) throw std::runtime_error("maxiter < 0");
  if (restart < 1 || restart > 1000) throw std::runtime_error("restart must be in [1, 1000]");
  const int m = restart;
  const bool pre = precond != 0;
  const size_t np = I.parts.size();
  load_rhs(b);
  I.launches = 0;
  std::vector<size_t> stride(np);
  for (size_t i = 0; i < np; ++i) {
    PartDev& pd = I.P(i);
    I.set_dev(pd);
    stride[i] = align_up((size_t)pd.lev[0]->n_own, 32);
    if (pd.gm_restart != m || pd.gm_precond != pre || pd.gm_basis.n == 0) {
      pd.gm_basis.alloc(stride[i] * (size_t)(pre ? 2 * m + 1 : m + 1), false);
      pd.gm_h.alloc((size_t)m + 2);
      pd.gm_restart = m;
      pd.gm_precond = pre;
    }
  }
  auto V = [&](size_t i, int j) { return I.P(i).gm_basis.p + stride[i] * (size_t)j; };
  auto Z = [&](size_t i, int j) { return pre ? I.P(i).gm_basis.p + stride[i] * (size_t)(m + 1 + j) : V(i, j); };
  const bool use_graph = I.h->opts.use_graph != 0;
  if (pre && use_graph && I.g_vcycle.empty()) capture(I.g_vcycle, &I.g_vcycle_nodes, [&] { enqueue_vcycle_entry(); });
  clear_done();
  // <u, v> over all parts, returned to the host (one synchronisation)
  auto host_dot = [&](auto&& uf, auto&& vf) {
    for (size_t i = 0; i < np; ++i) {
      PartDev& pd = I.P(i);
      I.set_dev(pd);
      const int n = (int)pd.lev[0]->n_own;
      k_dot<<<I.grid_red(n), BLOCK, 0, pd.stream>>>(uf(i), vf(i), n, pd.st.p, pd.partials.p, pd.rc, 3, 0);
      I.note_launch("k_dot");
    }
    for (size_t i = 0; i < np; ++i) {
      PartDev& pd = I.P(i);
      I.set_dev(pd);
      k_red_read<<<1, 1, 0, pd.stream>>>(pd.st.p, pd.rc, pd.scratch4.p);
      I.note_launch("k_red_read");
    }
    CK(cudaGetLastError());
    sync_all();
    double out[RED_W];
    I.set_dev(I.P(0));
    CK(cudaMemcpy(out, I.P(0).scratch4.p, sizeof(out), cudaMemcpyDeviceToHost));
    check_device_error();
    return out[3];
  };
  for (size_t i = 0; i < np; ++i) {
    PartDev& pd = I.P(i);
    I.set_dev(pd);
    CK(cudaEventRecord(pd.ev0, pd.stream));
    CK(cudaMemsetAsync(pd.xsol.p, 0, sizeof(double) * (size_t)pd.lev[0]->n_own, pd.stream));
  }
  // r lives in V_0 until it is normalised
  auto R = [&](size_t i) -> const double* { return V(i, 0); };
  for (size_t i = 0; i < np; ++i) {
    PartDev& pd = I.P(i);
    I.set_dev(pd);
    CK(cudaMemcpyAsync(V(i, 0), pd.bsave.p, sizeof(double) * (size_t)pd.lev[0]->n_own, cudaMemcpyDeviceToDevice, pd.stream));
  }
  const double beta0 = std::sqrt(host_dot(R, R));
  if (hist) hist[0] = beta0;
  int it = 0;
  bool done = (beta0 == 0.0 || maxiter == 0);
  std::vector<double> H((size_t)(m + 1) * m), cs(m), sn(m), g(m + 1), y(m), hcol(m + 2);
  double est = beta0;
  bool first = true;
  while (!done) {
    const double beta = first ? beta0 : std::sqrt(host_dot(R, R));
    first = false;
    for (size_t i = 0; i < np; ++i) {
      PartDev& pd = I.P(i);
      I.set_dev(pd);
      const int n = (int)pd.lev[0]->n_own;
      k_div<<<I.grid_for(n, BLOCK * 4), BLOCK, 0, pd.stream>>>(V(i, 0), V(i, 0), beta, n, pd.st.p);
      I.note_launch("k_div");
    }
    std::fill(H.begin(), H.end(), 0.0);
    std::fill(g.begin(), g.end(), 0.0);
    g[0] = beta;
    int j = 0;
    while (j < m) {
      if (pre) {  // z_j = M^-1 v_j
        for (size_t i = 0; i < np; ++i) {
          PartDev& pd = I.P(i);
          I.set_dev(pd);
          CK(cudaMemcpyAsync(pd.lev[0]->b.p, V(i, j), sizeof(double) * (size_t)pd.lev[0]->n_own, cudaMemcpyDeviceToDevice, pd.stream));
        }
        if (use_graph)
          launch_graphs(I.g_vcycle, I.g_vcycle_nodes);
        else
          enqueue_vcycle_entry();
        for (size_t i = 0; i < np; ++i) {
          PartDev& pd = I.P(i);
          I.set_dev(pd);
          CK(cudaMemcpyAsync(Z(i, j), pd.lev[0]->x.p, sizeof(double) * (size_t)pd.lev[0]->n_own, cudaMemcpyDeviceToDevice, pd.stream));
        }
      }
      {  // w = A z_j, into V_{j+1}
        std::vector<EpiArgs> epi(np);
        std::vector<const double*> xin(np);
        for (size_t i = 0; i < np; ++i) {
          xin[i] = Z(i, j);
          epi[i] = EpiArgs{V(i, j + 1), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
        }
        OpSpec op{0, PAMG_A_OO, 0, M_MUL, false, 0, false};
        enqueue_op(op, xin, epi);
      }
      for (int k = 0; k <= j + 1; ++k) {  // k <= j: h_kj = <w, v_k>, w -= h_kj v_k ; k = j + 1: h_{j+1,j} = ||w||, v_{j+1} = w / h
        for (size_t i = 0; i < np; ++i) {
          PartDev& pd = I.P(i);
          I.set_dev(pd);
          const int n = (int)pd.lev[0]->n_own;
          k_dot<<<I.grid_red(n), BLOCK, 0, pd.stream>>>(V(i, j + 1), k <= j ? V(i, k) : V(i, j + 1), n, pd.st.p, pd.partials.p, pd.rc, 3, 0);
          I.note_launch("k_dot");
        }
        for (size_t i = 0; i < np; ++i) {
          PartDev& pd = I.P(i);
          I.set_dev(pd);
          const int n = (int)pd.lev[0]->n_own;
          if (k <= j)
            k_gs_sub<<<I.grid_for(n, BLOCK * 4), BLOCK, 0, pd.stream>>>(V(i, j + 1), V(i, k), n, pd.st.p, pd.rc, pd.gm_h.p + k);
          else
            k_gs_norm<<<I.grid_for(n, BLOCK * 4), BLOCK, 0, pd.stream>>>(V(i, j + 1), n, pd.st.p, pd.rc, pd.gm_h.p + k);
          I.note_launch(k <= j ? "k_gs_sub" : "k_gs_norm");
        }
      }
      CK(cudaGetLastError());
      sync_all();
      I.set_dev(I.P(0));
      CK(cudaMemcpy(hcol.data(), I.P(0).gm_h.p, sizeof(double) * (size_t)(j + 2), cudaMemcpyDeviceToHost));
      check_device_error();
      for (int k = 0; k <= j + 1; ++k) H[(size_t)k * m + j] = hcol[k];
      for (int k = 0; k < j; ++k) {  // previous rotations on the new column
        const double t = cs[k] * H[(size_t)k * m + j] + sn[k] * H[(size_t)(k + 1) * m + j];
        H[(size_t)(k + 1) * m + j] = -sn[k] * H[(size_t)k * m + j] + cs[k] * H[(size_t)(k + 1) * m + j];
        H[(size_t)k * m + j] = t;
      }
      const double d = std::hypot(H[(size_t)j * m + j], H[(size_t)(j + 1) * m + j]);
      cs[j] = H[(size_t)j * m + j] / d;
      sn[j] = H[(size_t)(j + 1) * m + j] / d;
      H[(size_t)j * m + j] = d;
      H[(size_t)(j + 1) * m + j] = 0.0;
      g[j + 1] = -sn[j] * g[j];
      g[j] = cs[j] * g[j];
      ++j;
      ++it;
      est = std::fabs(g[j]);
      if (hist) hist[it] = est;
      if (est <= rtol * beta0 || it >= maxiter) {
        done = true;
        break;
      }
    }
    for (int i2 = j - 1; i2 >= 0; --i2) {  // back substitution
      double s2 = 0.0;
      for (int k = i2 + 1; k < j; ++k) s2 += H[(size_t)i2 * m + k] * y[k];
      y[i2] = (g[i2] - s2) / H[(size_t)i2 * m + i2];
    }
    for (int k = 0; k < j; ++k)  // x += y_k z_k, ascending k
      for (size_t i = 0; i < np; ++i) {
        PartDev& pd = I.P(i);
        I.set_dev(pd);
        const int n = (int)pd.lev[0]->n_own;
        k_axpy<<<I.grid_for(n, BLOCK * 4), BLOCK, 0, pd.stream>>>(pd.xsol.p, Z(i, k), y[k], n, pd.st.p);
        I.note_launch("k_axpy");
      }
    if (!done) {  // r = b - A x, into V_0
      std::vector<EpiArgs> epi(np);
      std::vector<const double*> xin(np);
      for (size_t i = 0; i < np; ++i) {
        xin[i] = I.P(i).xsol.p;
        epi[i] = EpiArgs{V(i, 0), I.P(i).bsave.p, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
      }
      OpSpec op{0, PAMG_A_OO, 0, M_RESID, false, 0, false};
      enqueue_op(op, xin, epi);
    }
  }
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaEventRecord(up->ev1, up->stream));
  }
  CK(cudaGetLastError());
  sync_all();
  float ms = 0, mx = 0;
  for (auto& up : I.parts) {
    I.set_dev(*up);
    CK(cudaEventElapsedTime(&ms, up->ev0, up->ev1));
    mx = std::max(mx, ms);
  }
  check_device_error();
  read_solution(x);
  const bool conv = est <= rtol * beta0;
  if (iters) *iters = it;
  I.stats.iters = it;
  I.stats.converged = conv;
  I.stats.r0_norm = beta0;
  I.stats.r_norm = est;
  I.stats.solve_ms = mx;
  I.stats.kernel_launches = I.launches;
  return conv ? PAMG_OK : PAMG_ERR_NOTCONV;
}

// ---------------------------------------------------------------------------------------------
// kernel timing hook (bench.py roofline leg)
// ---------------------------------------------------------------------------------------------
void Engine::time_kernel(int kind, int level, int reps, bool flush_l2, float* ms_out) {
  require_connected();
  Impl& I = *impl;
  if (level < 0 || level >= I.L) throw std::runtime_error("bad level");
  if ((kind == 2 || kind == 3) && level >= I.L - 1) throw std::runtime_error("no transfer operator on the coarsest level");
  PartDev& p0 = I.P(0);
  I.set_dev(p0);
  if (flush_l2 && !I.flush_buf) {
    I.flush_n = (size_t)(256u << 20) / sizeof(double);
    CK(cudaMalloc(&I.flush_buf, I.flush_n * sizeof(double)));
    CK(cudaMemset(I.flush_buf, 0, I.flush_n * sizeof(double)));
  }
  const size_t np = I.nslots();
  clear_done();
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  for (int r = 0; r < reps; ++r) {
    if (flush_l2) {
      I.set_dev(p0);
      k_flush<<<148 * 8, 256, 0, p0.stream>>>(I.flush_buf, I.flush_n);
    }
    I.set_dev(p0);
    CK(cudaEventRecord(e0, p0.stream));
    std::vector<EpiArgs> epi(np);
    if (kind == 0) {
      for (size_t i = 0; i < np; ++i)
        epi[i] = EpiArgs{I.S(i).lev[level]->t.p, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
      enqueue_op(OpSpec{level, PAMG_A_OO, level, M_MUL, false, 0, false}, ptrs(level, V_X), epi);
    } else if (kind == 1) {
      std::vector<double*> cur;
      for (size_t s = 0; s < np; ++s) cur.push_back(I.S(s).lev[level]->x.p);
      enqueue_smooth(level, 1, cur, false, false);
    } else if (kind == 2) {
      for (size_t i = 0; i < np; ++i) {
        LevelDev& ld = *I.S(i).lev[level];
        epi[i] = EpiArgs{ld.t.p, ld.b.p, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
      }
      enqueue_op(OpSpec{level, PAMG_A_OO, level, M_RESID, false, 0, false}, ptrs(level, V_X), epi);
      for (size_t i = 0; i < np; ++i) {
        LevelDev& lc = *I.S(i).lev[level + 1];
        epi[i] = EpiArgs{lc.b.p, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
      }
      enqueue_op(OpSpec{level, PAMG_R_OO, level, M_RESTRICT, false, 0, false}, ptrs(level, V_T), epi);
    } else if (kind == 3) {
      for (size_t i = 0; i < np; ++i) {
        LevelDev& ld = *I.S(i).lev[level];
        epi[i] = EpiArgs{ld.x2.p, ld.x.p, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0};
      }
      enqueue_op(OpSpec{level, PAMG_P_OO, level + 1, M_ADD, false, 0, false}, ptrs(level + 1, V_X), epi);
    } else if (kind == 4) {
      for (auto& up : I.parts) {
        PartDev& pd = *up;
        LevelDev& ld = *pd.lev[level];
        I.set_dev(pd);
        k_dot<<<I.grid_red(ld.n_own), BLOCK, 0, pd.stream>>>(ld.x.p, ld.b.p, (int)ld.n_own, pd.st.p, pd.partials.p, pd.rc, 3, 0);
      }
    } else if (kind == 8) {  // reference stream: read + write of the 256 MiB flush buffer (x += 1)
      if (!I.flush_buf) throw std::runtime_error("kind 8 needs flush_l2 != 0");
      k_flush<<<148 * 8, 256, 0, p0.stream>>>(I.flush_buf, I.flush_n);
    } else if (kind == 6) {  // SpMV with the fused p.q dot (as in the PCG iteration) + its reduce launch
      for (size_t i = 0; i < np; ++i) {
        LevelDev& ld = *I.S(i).lev[level];
        epi[i] = EpiArgs{ld.t.p, nullptr, nullptr, nullptr, nullptr, nullptr, ld.x.p, 0.0, 0.0};
      }
      enqueue_op(OpSpec{level, PAMG_A_OO, level, M_MUL, true, 3, false}, ptrs(level, V_X), epi);
    } else if (kind == 7) {  // Jacobi sweep with the fused r.z dot
      if (I.h->opts.smoother == PAMG_SMOOTHER_CHEBYSHEV) throw std::runtime_error("kind 7 needs a Jacobi smoother");
      std::vector<double*> cur;
      for (size_t s = 0; s < np; ++s) cur.push_back(I.S(s).lev[level]->x.p);
      enqueue_smooth(level, 1, cur, false, true);
    } else if (kind == 5) {
      const bool use_graph = I.h->opts.use_graph != 0;
      if (use_graph && I.g_vcycle.empty()) capture(I.g_vcycle, &I.g_vcycle_nodes, [&] { enqueue_vcycle_entry(); });
      if (use_graph)
        launch_graphs(I.g_vcycle, I.g_vcycle_nodes);
      else
        enqueue_vcycle_entry();
    } else {
      throw std::runtime_error("bad kernel kind");
    }
    I.set_dev(p0);
    CK(cudaEventRecord(e1, p0.stream));
    sync_all();
    CK(cudaEventElapsedTime(&ms_out[r], e0, e1));
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  check_device_error();
}

// ---------------------------------------------------------------------------------------------
// tracing: per-kernel start times (device globaltimer) of everything launched after trace_enable
// ---------------------------------------------------------------------------------------------
void Engine::trace_enable(int capacity) {
  Impl& I = *impl;
  sync_all();
  for (auto& up : I.parts) {
    PartDev& pd = *up;
    I.set_dev(pd);
    unsigned long long* buf = nullptr;
    uint32_t zero = 0, cap = 0;
    if (capacity > 0) {
      pd.trace.alloc((size_t)capacity);
      buf = pd.trace.p;
      cap = (uint32_t)capacity;
    }
    CK(cudaMemcpy(&pd.st.p->trace, &buf, sizeof(buf), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(&pd.st.p->trace_pos, &zero, sizeof(zero), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(&pd.st.p->trace_cap, &cap, sizeof(cap), cudaMemcpyHostToDevice));
  }
}

int Engine::trace_read(int part, unsigned long long* out, int cap) {
  Impl& I = *impl;
  if (part < 0 || part >= I.nparts || I.local_index[part] < 0) throw std::runtime_error("trace: part is not local");
  PartDev& pd = I.P(I.local_index[part]);
  sync_all();
  I.set_dev(pd);
  DevState s;
  CK(cudaMemcpy(&s, pd.st.p, sizeof(s), cudaMemcpyDeviceToHost));
  if (!s.trace) return 0;
  const int n = (int)std::min<uint32_t>(std::min<uint32_t>(s.trace_pos, s.trace_cap), (uint32_t)std::max(cap, 0));
  if (n > 0) CK(cudaMemcpy(out, pd.trace.p, (size_t)n * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  uint32_t zero = 0;
  CK(cudaMemcpy(&pd.st.p->trace_pos, &zero, sizeof(zero), cudaMemcpyHostToDevice));
  return n;
}

std::string Engine::trace_names() {
  std::string out;
  for (auto& n : impl->names) out += n + "\n";
  return out;
}

void Engine::get_stats(pamg_stats* s) {
  Impl& I = *impl;
  *s = I.stats;
  s->n_levels = I.L;
  s->fused_halo = I.fused_halo ? 1 : 0;
  s->tail_level = I.tail_level;
  auto fmt_of = [](const DevCsr& m) { return m.sell_rpt ? PAMG_FORMAT_SELL : m.stream ? PAMG_FORMAT_STREAM : PAMG_FORMAT_CSR; };
  for (int l = 0; l < 16; ++l) {
    const bool have = l < I.L && !I.parts.empty();
    s->format[l] = have ? fmt_of(I.P(0).lev[l]->blk[PAMG_A_OO]) : 0;
    s->format_p[l] = have && l + 1 < I.L ? fmt_of(I.P(0).lev[l]->blk[PAMG_P_OO]) : 0;
    s->format_r[l] = have && l + 1 < I.L ? fmt_of(I.P(0).lev[l]->blk[PAMG_R_OO]) : 0;
    s->lanes[l] = have ? I.P(0).lev[l]->blk[PAMG_A_OO].lanes : 0;
    s->sell_fill[l] = have ? I.P(0).lev[l]->blk[PAMG_A_OO].sell_fill : 1.0;
    s->value_indexed[l] = 0;
    if (have) {
      const LevelDev& ld = *I.P(0).lev[l];
      auto vi_of = [](const DevCsr& m) { return m.sell_vi || m.sell_vi4 || m.sell_diag; };
      auto wide_of = [](const DevCsr& m) { return m.sell_vi4 && m.vi4_ib == 2; };
      s->value_indexed[l] = (vi_of(ld.blk[PAMG_A_OO]) ? 1 : 0) | (vi_of(ld.blk[PAMG_P_OO]) ? 2 : 0) | (vi_of(ld.blk[PAMG_R_OO]) ? 4 : 0) |
                            (wide_of(ld.blk[PAMG_A_OO]) ? 8 : 0) | (wide_of(ld.blk[PAMG_P_OO]) ? 16 : 0) | (wide_of(ld.blk[PAMG_R_OO]) ? 32 : 0) |
                            (ld.blk[PAMG_A_OO].sell_diag ? 64 : 0);
    }
  }
}

}  // namespace pamg
