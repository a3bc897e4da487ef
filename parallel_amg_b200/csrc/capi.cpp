// capi.cpp — the C ABI of include/pamg.h: argument checking, exception -> status translation.
#include <omp.h>

#include <algorithm>
#include <cstring>
#include <memory>
#include <new>
#include <stdexcept>
#include <string>
#include <vector>

#include "engine.hpp"
#include "formats.hpp"
#include "host.hpp"

using namespace pamg;

struct pamg_ctx {
  int32_t nparts = 0;
  Csr A;                       // global matrix (host)
  std::vector<int32_t> owner;  // owner[gid]
  bool have_matrix = false;
  int32_t block_size = 1, ns_k = 0;   // DOFs per node / near-nullspace vectors (0: scalar smoothed aggregation)
  std::vector<double> nullspace;      // row-major n x ns_k
  std::vector<char> part_set;
  // rows staged by pamg_set_part_rows until all parts are in
  struct PartRows {
    std::vector<int64_t> own_to_global, rowptr, col;
    std::vector<double> val;
  };
  std::vector<PartRows> staged;
  Hierarchy h;
  int32_t ext_levels = 0;
  std::unique_ptr<Engine> eng;
  int32_t rhs_capacity = 1;  // for the next pamg_device_init
  std::string err;
};

namespace {

template <class F>
int guard(pamg_ctx* c, F&& f) {
  if (!c) return PAMG_ERR_ARG;
  try {
    c->err.clear();
    return f();
  } catch (const NoGpuError& e) {
    c->err = e.what();
    return PAMG_ERR_NOGPU;
  } catch (const CommError& e) {
    c->err = e.what();
    return PAMG_ERR_COMM;
  } catch (const CudaError& e) {
    c->err = e.what();
    return PAMG_ERR_CUDA;
  } catch (const std::bad_alloc&) {
    c->err = "out of host memory";
    return PAMG_ERR_ALLOC;
  } catch (const std::exception& e) {
    c->err = e.what();
    return PAMG_ERR_ARG;
  } catch (...) {
    c->err = "unknown error";
    return PAMG_ERR_ARG;
  }
}

void need(bool cond, const char* msg) {
  if (!cond) throw std::runtime_error(msg);
}

const PartLevel& part_level(pamg_ctx* c, int32_t level, int32_t part) {
  need(c->h.ready, "hierarchy not set up");
  need(level >= 0 && level < (int32_t)c->h.levels.size(), "bad level");
  need(part >= 0 && part < c->nparts, "bad part");
  return c->h.levels[level].parts[part];
}

Engine& engine(pamg_ctx* c) {
  if (!c->eng) throw std::runtime_error("device not initialised: call pamg_device_init");
  return *c->eng;
}

// the device state of a multi-column call: initialised with the capacity now set
Engine& engine_multi(pamg_ctx* c, int32_t k) {
  need(k >= 1 && k <= c->rhs_capacity, "k must be in 1..capacity (pamg_set_rhs_capacity)");
  Engine& e = engine(c);
  need(e.rhs_capacity() == c->rhs_capacity,
       "the right-hand-side capacity changed after pamg_device_init: call pamg_device_init again before a multi call");
  return e;
}

void merge_staged(pamg_ctx* c) {
  // all parts present: assemble the global CSR in gid order
  int64_t n = 0;
  for (auto& s : c->staged) n += (int64_t)s.own_to_global.size();
  c->owner.assign(n, -1);
  std::vector<int64_t> src_part(n), src_row(n);
  for (int32_t p = 0; p < c->nparts; ++p) {
    auto& s = c->staged[p];
    for (size_t i = 0; i < s.own_to_global.size(); ++i) {
      const int64_t g = s.own_to_global[i];
      need(g >= 0 && g < n, "own_to_global out of range");
      need(c->owner[g] < 0, "a global id is owned by two parts");
      need(i == 0 || s.own_to_global[i - 1] < g, "own_to_global must be ascending");
      c->owner[g] = p;
      src_part[g] = p;
      src_row[g] = (int64_t)i;
    }
  }
  Csr& A = c->A;
  A.nrows = A.ncols = n;
  A.ptr.assign(n + 1, 0);
  for (int64_t g = 0; g < n; ++g) {
    auto& s = c->staged[src_part[g]];
    A.ptr[g + 1] = A.ptr[g] + (s.rowptr[src_row[g] + 1] - s.rowptr[src_row[g]]);
  }
  huge_reserve(A.col, (size_t)A.ptr[n]);
  huge_reserve(A.val, (size_t)A.ptr[n]);
  A.col.resize(A.ptr[n]);
  A.val.resize(A.ptr[n]);
  for (int64_t g = 0; g < n; ++g) {
    auto& s = c->staged[src_part[g]];
    const int64_t b = s.rowptr[src_row[g]], e = s.rowptr[src_row[g] + 1];
    std::vector<std::pair<int64_t, double>> row;
    for (int64_t k = b; k < e; ++k) {
      need(s.col[k] >= 0 && s.col[k] < n, "column id out of range");
      row.emplace_back(s.col[k], s.val[k]);
    }
    std::sort(row.begin(), row.end(), [](const std::pair<int64_t, double>& x, const std::pair<int64_t, double>& y) { return x.first < y.first; });
    int64_t q = A.ptr[g];
    for (auto& e2 : row) {
      A.col[q] = e2.first;
      A.val[q++] = e2.second;
    }
  }
  c->staged.clear();
  c->staged.shrink_to_fit();
  c->have_matrix = true;
}

}  // namespace

extern "C" {

void pamg_default_options(pamg_options* o) {
  if (!o) return;
  std::memset(o, 0, sizeof(*o));
  o->struct_size = (int32_t)sizeof(pamg_options);
  o->eps_strength = 0.0;
  o->coarse_size = 500;
  o->max_levels = 12;
  o->smoother = PAMG_SMOOTHER_JACOBI;
  o->omega_jacobi = 2.0 / 3.0;
  o->nu_pre = 1;
  o->nu_post = 1;
  o->cheb_degree = 3;
  o->cheb_lo_frac = 1.0 / 30.0;
  o->cheb_hi_frac = 1.0;
  o->spmv_format = PAMG_FORMAT_AUTO;
  o->use_graph = 1;
  o->lanes_per_row = 0;
  o->tail_rows = 131072;
  o->sell_sigma = 0;
  o->sell_rows_per_thread = 0;
  o->fuse_halo = 1;
  o->cycle = PAMG_CYCLE_V;
}

int pamg_create(int32_t nparts, pamg_ctx** out) {
  if (!out || nparts < 1 || nparts > 256) return PAMG_ERR_ARG;
  try {
    pamg_ctx* c = new pamg_ctx;
    c->nparts = nparts;
    c->part_set.assign(nparts, 0);
    *out = c;
    return PAMG_OK;
  } catch (...) {
    return PAMG_ERR_ALLOC;
  }
}

void pamg_destroy(pamg_ctx* c) { delete c; }

const char* pamg_last_error(const pamg_ctx* c) { return c ? c->err.c_str() : "null context"; }

int pamg_set_part_rows(pamg_ctx* c, int32_t part, int64_t n_own, const int64_t* own_to_global, const int64_t* rowptr,
                       const int64_t* col_gid, const double* val) {
  return guard(c, [&] {
    need(part >= 0 && part < c->nparts, "bad part");
    need(n_own >= 0 && (n_own == 0 || (own_to_global && rowptr)), "null arrays");
    if (c->staged.empty()) c->staged.resize(c->nparts);
    auto& s = c->staged[part];
    s.own_to_global.assign(own_to_global, own_to_global + n_own);
    if (n_own) {
      need(rowptr[0] == 0, "rowptr must start at 0");
      for (int64_t i = 0; i < n_own; ++i) need(rowptr[i + 1] >= rowptr[i], "rowptr must be non-decreasing");
      s.rowptr.assign(rowptr, rowptr + n_own + 1);
      const int64_t nnz = rowptr[n_own];
      need(nnz == 0 || (col_gid && val), "null arrays");
      s.col.assign(col_gid, col_gid + nnz);
      s.val.assign(val, val + nnz);
    } else {
      s.rowptr.assign(1, 0);
    }
    c->part_set[part] = 1;
    c->have_matrix = false;
    bool all = true;
    for (char f : c->part_set) all = all && f;
    if (all) {
      merge_staged(c);
      c->part_set.assign(c->nparts, 0);
    }
    return PAMG_OK;
  });
}

int pamg_set_matrix_global(pamg_ctx* c, int64_t n, const int64_t* rowptr, const int64_t* col, const double* val,
                           const int32_t* owner) {
  return guard(c, [&] {
    need(n > 0 && rowptr && col && val && owner, "null arrays");
    need(rowptr[0] == 0, "rowptr must start at 0");
    for (int64_t i = 0; i < n; ++i) need(rowptr[i + 1] >= rowptr[i], "rowptr must be non-decreasing");
    Csr& A = c->A;
    A.nrows = A.ncols = n;
    A.ptr.assign(rowptr, rowptr + n + 1);
    const int64_t nnz = rowptr[n];
    A.col.assign(col, col + nnz);
    A.val.assign(val, val + nnz);
    for (int64_t i = 0; i < n; ++i)
      for (int64_t k = A.ptr[i]; k < A.ptr[i + 1]; ++k) {
        need(A.col[k] >= 0 && A.col[k] < n, "column id out of range");
        need(k == A.ptr[i] || A.col[k - 1] < A.col[k], "columns must be sorted and unique within a row");
      }
    c->owner.assign(owner, owner + n);
    for (int64_t i = 0; i < n; ++i) need(owner[i] >= 0 && owner[i] < c->nparts, "owner id out of range");
    c->have_matrix = true;
    return PAMG_OK;
  });
}

int pamg_gallery_poisson(pamg_ctx* c, int32_t ndim, const int64_t* nodes_per_dir, const int32_t* parts_per_dir) {
  return guard(c, [&] {
    need(ndim >= 1 && ndim <= 3 && nodes_per_dir && parts_per_dir, "bad arguments");
    int64_t np = 1;
    for (int a = 0; a < ndim; ++a) {
      need(nodes_per_dir[a] >= 1 && parts_per_dir[a] >= 1 && parts_per_dir[a] <= nodes_per_dir[a], "bad grid/partition");
      np *= parts_per_dir[a];
    }
    need(np == c->nparts, "prod(parts_per_dir) != nparts");
    gallery_poisson(ndim, nodes_per_dir, c->A);
    uniform_partition(ndim, nodes_per_dir, parts_per_dir, c->owner);
    c->have_matrix = true;
    return PAMG_OK;
  });
}

int pamg_gallery_diffusion_jump(pamg_ctx* c, int32_t ndim, const int64_t* nodes_per_dir, const int32_t* parts_per_dir,
                                int32_t blocks, double kmax, double eps_z) {
  return guard(c, [&] {
    need(ndim >= 1 && ndim <= 3 && nodes_per_dir && parts_per_dir && blocks >= 1, "bad arguments");
    int64_t np = 1;
    for (int a = 0; a < ndim; ++a) {
      need(nodes_per_dir[a] >= 1 && parts_per_dir[a] >= 1 && parts_per_dir[a] <= nodes_per_dir[a], "bad grid/partition");
      np *= parts_per_dir[a];
    }
    need(np == c->nparts, "prod(parts_per_dir) != nparts");
    gallery_diffusion_jump(ndim, nodes_per_dir, blocks, kmax, eps_z, c->A);
    uniform_partition(ndim, nodes_per_dir, parts_per_dir, c->owner);
    c->have_matrix = true;
    return PAMG_OK;
  });
}

int pamg_uniform_partition(int32_t ndim, const int64_t* nodes_per_dir, const int32_t* parts_per_dir, int32_t* owner_out) {
  if (ndim < 1 || ndim > 3 || !nodes_per_dir || !parts_per_dir || !owner_out) return PAMG_ERR_ARG;
  for (int a = 0; a < ndim; ++a)
    if (nodes_per_dir[a] < 1 || parts_per_dir[a] < 1 || parts_per_dir[a] > nodes_per_dir[a]) return PAMG_ERR_ARG;
  try {
    std::vector<int32_t> o;
    uniform_partition(ndim, nodes_per_dir, parts_per_dir, o);
    std::memcpy(owner_out, o.data(), o.size() * sizeof(int32_t));
    return PAMG_OK;
  } catch (...) {
    return PAMG_ERR_ARG;
  }
}

int pamg_host_matvec_global(pamg_ctx* c, const double* x, double* y) {
  return guard(c, [&] {
    need(c->have_matrix && x && y, "no matrix");
    matvec(c->A, x, y);
    return PAMG_OK;
  });
}

int pamg_global_size(pamg_ctx* c, int64_t* n, int64_t* nnz) {
  return guard(c, [&] {
    need(c->have_matrix, "no matrix");
    if (n) *n = c->A.nrows;
    if (nnz) *nnz = c->A.nnz();
    return PAMG_OK;
  });
}

void pamg_set_num_threads(int32_t n) { omp_set_num_threads(n > 0 ? n : omp_get_num_procs()); }

int pamg_setup(pamg_ctx* c, const pamg_options* o) {
  return guard(c, [&] {
    need(c->have_matrix, "no matrix: call pamg_set_part_rows / pamg_set_matrix_global / a gallery first");
    pamg_options opt;
    pamg_default_options(&opt);
    if (o) {
      need(o->struct_size == (int32_t)sizeof(pamg_options), "pamg_options.struct_size mismatch");
      opt = *o;
    }
    need(opt.coarse_size >= 1 && opt.max_levels >= 1 && opt.max_levels <= 16, "bad coarse_size/max_levels");
    need(opt.nu_pre >= 0 && opt.nu_post >= 0 && opt.nu_pre + opt.nu_post >= 0, "bad sweep counts");
    need(opt.smoother >= 0 && opt.smoother <= 2, "bad smoother");
    need(opt.cycle == PAMG_CYCLE_V || opt.cycle == PAMG_CYCLE_W, "bad cycle");
    c->eng.reset();
    if (c->ns_k > 0) need((int64_t)c->nullspace.size() == c->A.nrows * c->ns_k, "near-nullspace does not match the matrix");
    build_hierarchy(c->A, c->owner, c->nparts, opt, c->h, c->block_size, c->ns_k, c->ns_k > 0 ? &c->nullspace : nullptr);
    return PAMG_OK;
  });
}

// ---- device-layout queries (host-side conversions of formats.hpp; no GPU needed) ------------------------
int pamg_layout_sell(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int32_t rows_per_slice, int32_t sigma,
                     int64_t* n_slices, int64_t* stored, int32_t* permuted, int32_t* slice_off, int32_t* col, double* val,
                     int32_t* perm) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    need(which == PAMG_A_OO || which == PAMG_P_OO || which == PAMG_R_OO, "SELL applies to own-own blocks");
    need(rows_per_slice >= 1 && rows_per_slice <= 1024 && n_slices && stored && permuted, "bad arguments");
    SellHost sh;
    const int inter = sigma < 0 ? -sigma : 0;  // sigma = -R: the interleaved layout (R rows per lane, rows_per_slice = 32 R)
    sell_layout(pl.blk[which], rows_per_slice, inter ? 1 : sigma, sh, col != nullptr || val != nullptr, inter);
    const int64_t ns = (int64_t)sh.off.size() - 1;
    *n_slices = ns;
    *stored = (int64_t)sh.off[ns] * rows_per_slice;
    *permuted = sh.permuted ? 1 : 0;
    if (slice_off) std::memcpy(slice_off, sh.off.data(), sh.off.size() * sizeof(int32_t));
    if (col) std::memcpy(col, sh.col.data(), (size_t)*stored * sizeof(int32_t));
    if (val) std::memcpy(val, sh.val.data(), (size_t)*stored * sizeof(double));
    if (perm) std::memcpy(perm, sh.perm.data(), sh.perm.size() * sizeof(int32_t));
    return PAMG_OK;
  });
}

int pamg_layout_sell_values(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int32_t rows_per_slice, int32_t sigma,
                            int32_t* indexed, int64_t* stored, double* dict, uint8_t* vidx) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    need(which == PAMG_A_OO || which == PAMG_P_OO || which == PAMG_R_OO, "SELL applies to own-own blocks");
    need(rows_per_slice >= 1 && rows_per_slice <= 1024 && indexed && stored, "bad arguments");
    SellHost sh;
    int ib = value_dictionary(pl.blk[which], sh.dict, 255) ? 1 : 0;
    if (!ib && value_dictionary(pl.blk[which], sh.dict, 4095)) ib = 2;  // the wide form of the 128-row kernel
    *indexed = ib;
    const int inter = sigma < 0 ? -sigma : 0;
    sell_layout(pl.blk[which], rows_per_slice, inter ? 1 : sigma, sh, ib && vidx != nullptr, inter);
    *stored = (int64_t)sh.off[sh.off.size() - 1] * rows_per_slice;
    if (!ib) return PAMG_OK;
    if (dict) {
      std::memset(dict, 0, 4096 * sizeof(double));
      std::memcpy(dict, sh.dict.data(), sh.dict.size() * sizeof(double));
    }
    if (vidx) {
      sell_value_index(sh, ib);
      std::memcpy(vidx, sh.vidx.data(), (size_t)*stored * (size_t)ib);
    }
    return PAMG_OK;
  });
}

int pamg_layout_sell_diag(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int32_t* ndiag, int32_t* off, int64_t* stored,
                          double* dict, uint8_t* idx) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    need(which == PAMG_A_OO || which == PAMG_P_OO || which == PAMG_R_OO, "SELL applies to own-own blocks");
    need(ndiag && stored, "bad arguments");
    DiagHost dh;
    *ndiag = 0;
    *stored = 0;
    if (which != PAMG_A_OO || !diag_layout(pl.blk[which], dh, idx != nullptr)) return PAMG_OK;  // the upload takes it for A only
    *ndiag = (int32_t)dh.off.size();
    *stored = dh.nslices * (int64_t)dh.off.size() * 128;
    if (off) std::memcpy(off, dh.off.data(), dh.off.size() * sizeof(int32_t));
    if (dict) std::memcpy(dict, dh.dict.data(), 256 * sizeof(double));
    if (idx) std::memcpy(idx, dh.idx.data(), dh.idx.size());
    return PAMG_OK;
  });
}

int pamg_layout_stream(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int32_t max_rows, int32_t max_entries,
                       int64_t* n_blocks, int32_t* first_row, int32_t* first_entry) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    need(which == PAMG_A_OO || which == PAMG_P_OO || which == PAMG_R_OO, "CSR-stream applies to own-own blocks");
    need(max_rows >= 1 && max_entries >= 1 && n_blocks, "bad arguments");
    std::vector<std::pair<int32_t, int32_t>> blk;
    if (!stream_row_blocks(pl.blk[which], max_rows, max_entries, blk)) {
      *n_blocks = -1;  // a row exceeds the buffer: the block keeps the sub-warp CSR kernel
      return PAMG_OK;
    }
    *n_blocks = (int64_t)blk.size() - 1;
    for (size_t k = 0; k < blk.size(); ++k) {
      if (first_row) first_row[k] = blk[k].first;
      if (first_entry) first_entry[k] = blk[k].second;
    }
    return PAMG_OK;
  });
}

int pamg_layout_boundary(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int64_t* n_rows, int64_t* n_entries,
                         int32_t* lanes, int32_t* rows, int32_t* ptr, int32_t* mid, int32_t* col, double* val, uint8_t* skip) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    need(which == PAMG_A_OO || which == PAMG_P_OO || which == PAMG_R_OO, "pass the own-own block id");
    need(n_rows && n_entries && lanes, "bad arguments");
    BndHost hb;
    bnd_layout(pl.blk[which], pl.blk[which + 1], hb);
    *n_rows = (int64_t)hb.rows.size();
    *n_entries = (int64_t)hb.col.size();
    *lanes = hb.lanes;
    if (rows) std::memcpy(rows, hb.rows.data(), hb.rows.size() * sizeof(int32_t));
    if (ptr) std::memcpy(ptr, hb.ptr.data(), hb.ptr.size() * sizeof(int32_t));
    if (mid) std::memcpy(mid, hb.mid.data(), hb.mid.size() * sizeof(int32_t));
    if (col) std::memcpy(col, hb.col.data(), hb.col.size() * sizeof(int32_t));
    if (val) std::memcpy(val, hb.val.data(), hb.val.size() * sizeof(double));
    if (skip) std::memcpy(skip, hb.skip.data(), (size_t)pl.blk[which].nrows);
    return PAMG_OK;
  });
}

int pamg_hierarchy_save(pamg_ctx* c, const char* path) {
  return guard(c, [&] {
    need(path != nullptr, "null path");
    need(c->h.ready, "hierarchy not set up");
    save_hierarchy(c->h, path);
    return PAMG_OK;
  });
}

int pamg_hierarchy_load(pamg_ctx* c, const char* path, int32_t keep_part) {
  return guard(c, [&] {
    need(path != nullptr, "null path");
    c->eng.reset();
    load_hierarchy(c->h, path, keep_part);
    need(c->h.nparts == c->nparts, "hierarchy file was written for a different number of parts");
    return PAMG_OK;
  });
}

int pamg_set_near_nullspace(pamg_ctx* c, int32_t block_size, int32_t k, const double* B) {
  return guard(c, [&] {
    need(c->have_matrix, "set the matrix first");
    if (k <= 0 || !B) {  // back to scalar smoothed aggregation
      c->block_size = 1;
      c->ns_k = 0;
      c->nullspace.clear();
      return PAMG_OK;
    }
    need(block_size >= 1 && k <= 64 && c->A.nrows % block_size == 0, "bad block size / vector count");
    c->block_size = block_size;
    c->ns_k = k;
    c->nullspace.assign(B, B + (size_t)c->A.nrows * k);
    return PAMG_OK;
  });
}

int pamg_gallery_elasticity(pamg_ctx* c, const int64_t* nodes_per_dir, const int32_t* parts_per_dir, double E, double nu) {
  return guard(c, [&] {
    need(nodes_per_dir && parts_per_dir, "bad arguments");
    int64_t np = 1;
    for (int a = 0; a < 3; ++a) {
      need(nodes_per_dir[a] >= 1 && parts_per_dir[a] >= 1 && parts_per_dir[a] <= nodes_per_dir[a], "bad grid/partition");
      np *= parts_per_dir[a];
    }
    need(np == c->nparts, "prod(parts_per_dir) != nparts");
    need(E > 0.0 && nu > -1.0 && nu < 0.5, "bad material constants");
    std::vector<double> coords;
    gallery_elasticity(nodes_per_dir, E, nu, c->A, coords);
    std::vector<int32_t> node_owner;
    uniform_partition(3, nodes_per_dir, parts_per_dir, node_owner);
    c->owner.resize(node_owner.size() * 3);
    for (size_t v = 0; v < node_owner.size(); ++v) c->owner[3 * v] = c->owner[3 * v + 1] = c->owner[3 * v + 2] = node_owner[v];
    rigid_body_modes(coords, c->nullspace);
    c->block_size = 3;
    c->ns_k = 6;
    c->have_matrix = true;
    return PAMG_OK;
  });
}

int pamg_get_near_nullspace(pamg_ctx* c, int32_t* block_size, int32_t* k, double* B /* may be NULL */) {
  return guard(c, [&] {
    need(block_size && k, "null output");
    *block_size = c->block_size;
    *k = c->ns_k;
    if (B && c->ns_k > 0) std::memcpy(B, c->nullspace.data(), c->nullspace.size() * sizeof(double));
    return PAMG_OK;
  });
}

int pamg_hierarchy_begin(pamg_ctx* c, int32_t n_levels, const pamg_options* o) {
  return guard(c, [&] {
    need(n_levels >= 1 && n_levels <= 16, "bad level count");
    pamg_options opt;
    pamg_default_options(&opt);
    if (o) {
      need(o->struct_size == (int32_t)sizeof(pamg_options), "pamg_options.struct_size mismatch");
      opt = *o;
    }
    c->eng.reset();
    c->h = Hierarchy();
    c->h.nparts = c->nparts;
    c->h.opts = opt;
    c->h.levels.resize(n_levels);
    for (auto& l : c->h.levels) l.parts.resize(c->nparts);
    c->ext_levels = n_levels;
    return PAMG_OK;
  });
}

int pamg_level_upload(pamg_ctx* c, int32_t level, int32_t part, int64_t n_own, int64_t n_ghost, const int64_t* own_to_global,
                      const int64_t* ghost_to_global, const int32_t* ghost_to_owner, int64_t n_own_coarse,
                      int64_t n_ghost_coarse, const int64_t* const rowptr[6], const int32_t* const col[6],
                      const double* const val[6], double rho) {
  return guard(c, [&] {
    need(c->ext_levels > 0 && level >= 0 && level < c->ext_levels, "pamg_hierarchy_begin first / bad level");
    need(part >= 0 && part < c->nparts, "bad part");
    need(n_own >= 0 && n_ghost >= 0 && n_own < INT32_MAX && n_ghost < INT32_MAX, "bad sizes");
    need((n_own == 0 || own_to_global) && (n_ghost == 0 || (ghost_to_global && ghost_to_owner)), "null index maps");
    need(rowptr && col && val, "null block tables");
    PartLevel& pl = c->h.levels[level].parts[part];
    pl = PartLevel();
    pl.present = true;
    pl.n_own = n_own;
    pl.n_ghost = n_ghost;
    pl.n_own_coarse = n_own_coarse;
    pl.n_ghost_coarse = n_ghost_coarse;
    pl.own_to_global.assign(own_to_global, own_to_global + n_own);
    pl.ghost_to_global.assign(ghost_to_global, ghost_to_global + n_ghost);
    pl.ghost_to_owner.assign(ghost_to_owner, ghost_to_owner + n_ghost);
    c->h.levels[level].rho = rho;
    const bool last = (level == c->ext_levels - 1);
    for (int b = 0; b < 6; ++b) {
      if (last && b >= PAMG_P_OO) continue;
      const bool is_r = (b >= PAMG_R_OO);
      const int64_t nr = is_r ? n_own_coarse : n_own;
      int64_t nc;
      if (b == PAMG_A_OO || b == PAMG_R_OO) nc = n_own;
      else if (b == PAMG_A_OG || b == PAMG_R_OG) nc = n_ghost;
      else if (b == PAMG_P_OO) nc = n_own_coarse;
      else nc = n_ghost_coarse;
      LocalCsr& m = pl.blk[b];
      m.nrows = nr;
      m.ncols = nc;
      if (!rowptr[b]) {
        need((b & 1) == 1, "own-own blocks are mandatory");
        m.ptr.assign(nr + 1, 0);
        continue;
      }
      m.ptr.assign(rowptr[b], rowptr[b] + nr + 1);
      need(m.ptr[0] == 0, "rowptr must start at 0");
      const int64_t nnz = m.ptr[nr];
      need(nnz == 0 || (col[b] && val[b]), "null block arrays");
      need(nnz < INT32_MAX, "block too large");
      m.col.assign(col[b], col[b] + nnz);
      m.val.assign(val[b], val[b] + nnz);
      for (int64_t k = 0; k < nnz; ++k) need(m.col[k] >= 0 && m.col[k] < nc, "local column out of range");
    }
    return PAMG_OK;
  });
}

int pamg_coarse_upload(pamg_ctx* c, int64_t n, const double* inverse_row_major) {
  return guard(c, [&] {
    need(c->ext_levels > 0 && n >= 1 && n <= 8192 && inverse_row_major, "bad arguments");
    c->h.n_coarse = n;
    c->h.coarse_inv.assign(inverse_row_major, inverse_row_major + n * n);
    return PAMG_OK;
  });
}

int pamg_hierarchy_end(pamg_ctx* c) {
  return guard(c, [&] {
    need(c->ext_levels > 0, "pamg_hierarchy_begin first");
    finalize_external(c->h);
    return PAMG_OK;
  });
}

int pamg_num_levels(pamg_ctx* c, int32_t* n_levels) {
  return guard(c, [&] {
    need(c->h.ready && n_levels, "hierarchy not set up");
    *n_levels = (int32_t)c->h.levels.size();
    return PAMG_OK;
  });
}

int pamg_get_level_info(pamg_ctx* c, int32_t level, int32_t part, pamg_level_info* info) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(info != nullptr, "null info");
    std::memset(info, 0, sizeof(*info));
    info->n_global = c->h.levels[level].n_global;
    info->n_own = pl.n_own;
    info->n_ghost = pl.n_ghost;
    info->n_own_coarse = pl.n_own_coarse;
    for (int b = 0; b < 6; ++b) info->nnz[b] = pl.block_nnz(b);
    info->n_recv_nbrs = (int32_t)pl.recv.size();
    info->n_send_nbrs = (int32_t)pl.send.size();
    info->n_send = pl.n_send_entries();
    info->rho = c->h.levels[level].rho;
    info->omega_p = c->h.levels[level].omega_p;
    return PAMG_OK;
  });
}

int pamg_get_index_maps(pamg_ctx* c, int32_t level, int32_t part, int64_t* own_to_global, int64_t* ghost_to_global,
                        int32_t* ghost_to_owner) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    if (own_to_global) std::memcpy(own_to_global, pl.own_to_global.data(), pl.n_own * sizeof(int64_t));
    if (ghost_to_global) std::memcpy(ghost_to_global, pl.ghost_to_global.data(), pl.n_ghost * sizeof(int64_t));
    if (ghost_to_owner) std::memcpy(ghost_to_owner, pl.ghost_to_owner.data(), pl.n_ghost * sizeof(int32_t));
    return PAMG_OK;
  });
}

int pamg_get_block(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int64_t* rowptr, int32_t* col, double* val) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    need(which >= 0 && which < 6, "bad block id");
    const LocalCsr& m = pl.blk[which];
    if (rowptr && !m.ptr.empty()) std::memcpy(rowptr, m.ptr.data(), m.ptr.size() * sizeof(int64_t));
    if (col && m.nnz()) std::memcpy(col, m.col.data(), m.nnz() * sizeof(int32_t));
    if (val && m.nnz()) std::memcpy(val, m.val.data(), m.nnz() * sizeof(double));
    return PAMG_OK;
  });
}

int pamg_get_aggregates(pamg_ctx* c, int32_t level, int32_t part, int32_t* agg_local) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    need((int64_t)pl.agg_local.size() == pl.n_own && agg_local, "no aggregates on this level");
    std::memcpy(agg_local, pl.agg_local.data(), pl.n_own * sizeof(int32_t));
    return PAMG_OK;
  });
}

int pamg_get_halo_plan(pamg_ctx* c, int32_t level, int32_t part, int32_t* recv_part, int32_t* recv_slot0, int32_t* recv_count,
                       int32_t* send_part, int32_t* send_slot0, int32_t* send_count, int32_t* send_idx) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    for (size_t k = 0; k < pl.recv.size(); ++k) {
      if (recv_part) recv_part[k] = pl.recv[k].part;
      if (recv_slot0) recv_slot0[k] = pl.recv[k].slot0;
      if (recv_count) recv_count[k] = pl.recv[k].count;
    }
    for (size_t k = 0; k < pl.send.size(); ++k) {
      if (send_part) send_part[k] = pl.send[k].part;
      if (send_slot0) send_slot0[k] = pl.send[k].slot0;
      if (send_count) send_count[k] = pl.send[k].count;
    }
    if (send_idx && !pl.send_idx.empty()) std::memcpy(send_idx, pl.send_idx.data(), pl.send_idx.size() * sizeof(int32_t));
    return PAMG_OK;
  });
}

int pamg_get_coarse_inverse(pamg_ctx* c, int64_t* n, double* inverse_row_major) {
  return guard(c, [&] {
    need(c->h.ready, "hierarchy not set up");
    if (n) *n = c->h.n_coarse;
    if (inverse_row_major) std::memcpy(inverse_row_major, c->h.coarse_inv.data(), c->h.coarse_inv.size() * sizeof(double));
    return PAMG_OK;
  });
}

int pamg_get_diag(pamg_ctx* c, int32_t level, int32_t part, double* diag, double* diag_l1) {
  return guard(c, [&] {
    const PartLevel& pl = part_level(c, level, part);
    need(pl.full, "this part was loaded as metadata only (pamg_hierarchy_load keep_part)");
    if (diag) std::memcpy(diag, pl.diag.data(), pl.n_own * sizeof(double));
    if (diag_l1) std::memcpy(diag_l1, pl.diag_l1.data(), pl.n_own * sizeof(double));
    return PAMG_OK;
  });
}

// ---- device ------------------------------------------------------------------------------------
int pamg_device_init(pamg_ctx* c, int32_t nlocal, const int32_t* local_parts, const int32_t* device_ids) {
  return guard(c, [&] {
    need(c->h.ready, "hierarchy not set up");
    need(nlocal >= 1 && nlocal <= c->nparts && local_parts, "bad local part list");
    c->eng.reset();
    c->eng.reset(new Engine(&c->h, nlocal, local_parts, device_ids, c->rhs_capacity));
    return PAMG_OK;
  });
}

int pamg_set_rhs_capacity(pamg_ctx* c, int32_t kmax) {
  return guard(c, [&] {
    need(kmax >= 1 && kmax <= PAMG_MAX_RHS, "right-hand-side capacity must be in 1..PAMG_MAX_RHS (8)");
    c->rhs_capacity = kmax;
    return PAMG_OK;
  });
}

int pamg_set_kernel_options(pamg_ctx* c, const pamg_options* o) {
  return guard(c, [&] {
    need(o && o->struct_size == (int32_t)sizeof(pamg_options), "bad options struct");
    need(c->h.ready, "hierarchy not set up");
    c->h.opts.spmv_format = o->spmv_format;
    c->h.opts.lanes_per_row = o->lanes_per_row;
    c->h.opts.use_graph = o->use_graph;
    c->h.opts.sell_sigma = o->sell_sigma;
    c->h.opts.sell_rows_per_thread = o->sell_rows_per_thread;
    c->h.opts.fuse_halo = o->fuse_halo;
    c->h.opts.tail_rows = o->tail_rows;
    return PAMG_OK;
  });
}

int32_t pamg_comm_handle_bytes(void) { return Engine::handle_bytes(); }

int pamg_comm_export(pamg_ctx* c, int32_t local_part, void* blob) {
  return guard(c, [&] {
    need(blob != nullptr, "null blob");
    engine(c).export_handle(local_part, blob);
    return PAMG_OK;
  });
}
int pamg_comm_import(pamg_ctx* c, int32_t remote_part, const void* blob) {
  return guard(c, [&] {
    need(blob != nullptr, "null blob");
    engine(c).import_handle(remote_part, blob);
    return PAMG_OK;
  });
}
int pamg_comm_connect(pamg_ctx* c) {
  return guard(c, [&] {
    engine(c).connect();
    return PAMG_OK;
  });
}

int pamg_spmv(pamg_ctx* c, int32_t level, const double* const* x, double* const* y) {
  return guard(c, [&] {
    need(x && y, "null vectors");
    engine(c).spmv(level, x, y);
    return PAMG_OK;
  });
}
int pamg_consistent(pamg_ctx* c, int32_t level, double* const* v) {
  return guard(c, [&] {
    need(v != nullptr, "null vectors");
    engine(c).consistent(level, v);
    return PAMG_OK;
  });
}
int pamg_assemble(pamg_ctx* c, int32_t level, double* const* v) {
  return guard(c, [&] {
    need(v != nullptr, "null vectors");
    engine(c).assemble(level, v);
    return PAMG_OK;
  });
}
int pamg_smooth(pamg_ctx* c, int32_t level, int32_t nu, const double* const* b, double* const* x) {
  return guard(c, [&] {
    need(b && x && nu >= 0, "bad arguments");
    engine(c).smooth(level, nu, b, x);
    return PAMG_OK;
  });
}
int pamg_residual_restrict(pamg_ctx* c, int32_t level, const double* const* b, const double* const* x, double* const* r,
                           double* const* bc) {
  return guard(c, [&] {
    need(b && x && bc, "null vectors");
    engine(c).residual_restrict(level, b, x, r, bc);
    return PAMG_OK;
  });
}
int pamg_prolong_correct(pamg_ctx* c, int32_t level, const double* const* ec, double* const* x) {
  return guard(c, [&] {
    need(ec && x, "null vectors");
    engine(c).prolong_correct(level, ec, x);
    return PAMG_OK;
  });
}
int pamg_dot(pamg_ctx* c, int32_t level, const double* const* u, const double* const* v, double* out) {
  return guard(c, [&] {
    need(u && v && out, "null arguments");
    *out = engine(c).dot(level, u, v);
    return PAMG_OK;
  });
}
int pamg_vcycle(pamg_ctx* c, const double* const* b, double* const* x) {
  return guard(c, [&] {
    need(b && x, "null vectors");
    engine(c).vcycle(b, x);
    return PAMG_OK;
  });
}
int pamg_pcg(pamg_ctx* c, const double* const* b, double* const* x, double rtol, int32_t maxiter, int32_t precond,
             int32_t* iters, double* resid_hist) {
  return guard(c, [&] {
    need(b && x && rtol >= 0.0 && maxiter >= 0, "bad arguments");
    return engine(c).pcg(b, x, rtol, maxiter, precond != 0 ? 1 : 0, iters, resid_hist);
  });
}
int pamg_fcg(pamg_ctx* c, const double* const* b, double* const* x, double rtol, int32_t maxiter, int32_t* iters,
             double* resid_hist) {
  return guard(c, [&] {
    need(b && x && rtol >= 0.0 && maxiter >= 0, "bad arguments");
    return engine(c).pcg(b, x, rtol, maxiter, 2, iters, resid_hist);
  });
}
int pamg_spmv_multi(pamg_ctx* c, int32_t level, int32_t k, const double* const* x, double* const* y) {
  return guard(c, [&] {
    need(x && y, "null vectors");
    engine_multi(c, k).spmv_multi(level, k, x, y);
    return PAMG_OK;
  });
}
int pamg_vcycle_multi(pamg_ctx* c, int32_t k, const double* const* b, double* const* x) {
  return guard(c, [&] {
    need(b && x, "null vectors");
    engine_multi(c, k).vcycle_multi(k, b, x);
    return PAMG_OK;
  });
}
int pamg_pcg_multi(pamg_ctx* c, int32_t k, const double* const* b, double* const* x, double rtol, int32_t maxiter, int32_t mode,
                   int32_t* iters, int32_t* converged, double* resid_hist) {
  return guard(c, [&] {
    need(b && x && rtol >= 0.0 && maxiter >= 0 && mode >= 0 && mode <= 2, "bad arguments");
    return engine_multi(c, k).pcg_multi(k, b, x, rtol, maxiter, mode, iters, converged, resid_hist);
  });
}
int pamg_time_kernel_multi(pamg_ctx* c, int32_t k, int32_t kind, int32_t level, int32_t reps, int32_t flush_l2, float* ms_out) {
  return guard(c, [&] {
    need(reps >= 1 && ms_out, "bad arguments");
    engine_multi(c, k).time_kernel_multi(k, kind, level, reps, flush_l2 != 0, ms_out);
    return PAMG_OK;
  });
}
int pamg_fgmres(pamg_ctx* c, const double* const* b, double* const* x, double rtol, int32_t maxiter, int32_t restart,
                int32_t precond, int32_t* iters, double* resid_hist) {
  return guard(c, [&] {
    need(b && x && rtol >= 0.0 && maxiter >= 0 && restart >= 1, "bad arguments");
    return engine(c).fgmres(b, x, rtol, maxiter, restart, precond, iters, resid_hist);
  });
}
int pamg_load_rhs(pamg_ctx* c, const double* const* b) {
  return guard(c, [&] {
    need(b != nullptr, "null vectors");
    engine(c).load_rhs(b);
    return PAMG_OK;
  });
}
int pamg_pcg_resident(pamg_ctx* c, double rtol, int32_t maxiter, int32_t precond, int32_t* iters, double* resid_hist) {
  return guard(c, [&] {
    need(rtol >= 0.0 && maxiter >= 0, "bad arguments");
    return engine(c).pcg_resident(rtol, maxiter, precond != 0 ? 1 : 0, iters, resid_hist);
  });
}
int pamg_read_solution(pamg_ctx* c, double* const* x) {
  return guard(c, [&] {
    need(x != nullptr, "null vectors");
    engine(c).read_solution(x);
    return PAMG_OK;
  });
}
int pamg_time_kernel(pamg_ctx* c, int32_t kind, int32_t level, int32_t reps, int32_t flush_l2, float* ms_out) {
  return guard(c, [&] {
    need(reps >= 1 && ms_out, "bad arguments");
    engine(c).time_kernel(kind, level, reps, flush_l2 != 0, ms_out);
    return PAMG_OK;
  });
}
int pamg_trace_enable(pamg_ctx* c, int32_t capacity) {
  return guard(c, [&] {
    engine(c).trace_enable(capacity);
    return PAMG_OK;
  });
}
int pamg_trace_read(pamg_ctx* c, int32_t part, uint64_t* out, int32_t cap, int32_t* n) {
  return guard(c, [&] {
    need(out && n, "null output");
    *n = engine(c).trace_read(part, (unsigned long long*)out, cap);
    return PAMG_OK;
  });
}
int pamg_trace_names(pamg_ctx* c, char* buf, int32_t cap) {
  return guard(c, [&] {
    need(buf && cap > 0, "null buffer");
    const std::string s = engine(c).trace_names();
    std::strncpy(buf, s.c_str(), (size_t)cap - 1);
    buf[cap - 1] = 0;
    return PAMG_OK;
  });
}

int pamg_get_stats(pamg_ctx* c, pamg_stats* s) {
  return guard(c, [&] {
    need(s != nullptr, "null stats");
    engine(c).get_stats(s);
    return PAMG_OK;
  });
}

}  // extern "C"
