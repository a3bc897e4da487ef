// formats.hpp — host-side conversion of a split-format block (LocalCsr) into the device layouts of
// kernels.cuh: SELL-C-sigma slices, CSR-stream row blocks, boundary-row lists.  Host-only and header-only so
// that engine.cu (upload) and the C ABI's layout queries (CPU-testable invariants) share one implementation.
#pragma once
#include <algorithm>
#include <climits>
#include <cstring>
#include <cstdint>
#include <stdexcept>
#include <utility>
#include <vector>

#include "host.hpp"

namespace pamg {

// ---- SELL-C-sigma --------------------------------------------------------------------------------------
// C rows per slice; rows sorted by length (descending, stable) inside windows of `sigma` rows (sigma <= 1: no
// sorting); slice sl stores width(sl) = max row length entries per row, column-major: entry j of slot q lives
// at (off[sl] + j) * C + q.  Padding = (0.0, last column of the row) so that a gather stays in range.
struct SellHost {
  std::vector<int32_t> off, col, perm;  // off: [nslices + 1] in units of C entries; perm: slot -> row
  std::vector<double> val;
  bool permuted = false;
  double fill = 1.0;  // stored entries / nnz
  // value-indexed storage (kernels.cuh k_spmv_sell_vi): dict = the distinct values (dict[0] = +0.0, the padding value; 256
  // entries, unused ones 0.0), vidx = one byte per stored entry, same layout as col.  Empty when the operator has more
  // than 255 distinct non-padding values.
  std::vector<double> dict;
  std::vector<uint8_t> vidx;
};

// Distinct values of m by BIT PATTERN (-0.0 and +0.0 are different entries: the products keep their sign), ascending by
// pattern behind dict[0] = +0.0.  Returns false as soon as more than 255 are seen (then `dict` is empty).
inline bool value_dictionary(const LocalCsr& m, std::vector<double>& dict, int max_distinct = 255) {
  dict.clear();
  const int64_t nnz = m.nnz();
  auto bits = [](double v) {
    uint64_t b;
    std::memcpy(&b, &v, sizeof(b));
    return b;
  };
  std::vector<uint64_t> all;
  bool too_many = false;
#pragma omp parallel
  {
    std::vector<uint64_t> mine;  // sorted, tiny
    uint64_t last = ~0ull;       // no finite double: a NaN pattern that never occurs as a stored value twice in a row first
    bool have_last = false;
#pragma omp for schedule(static)
    for (int64_t k = 0; k < nnz; ++k) {
      bool stop;
#pragma omp atomic read
      stop = too_many;
      if (stop) continue;
      const uint64_t b = bits(m.val[k]);
      if (have_last && b == last) continue;
      last = b;
      have_last = true;
      auto it = std::lower_bound(mine.begin(), mine.end(), b);
      if (it == mine.end() || *it != b) {
        mine.insert(it, b);
        if ((int)mine.size() > max_distinct) {
#pragma omp atomic write
          too_many = true;
        }
      }
    }
#pragma omp critical
    all.insert(all.end(), mine.begin(), mine.end());
  }
  if (too_many) return false;
  std::sort(all.begin(), all.end());
  all.erase(std::unique(all.begin(), all.end()), all.end());
  all.erase(std::remove(all.begin(), all.end(), (uint64_t)0), all.end());  // +0.0 is dict[0] anyway
  if ((int)all.size() > max_distinct) return false;
  dict.assign(max_distinct <= 255 ? 256 : all.size() + 1, 0.0);  // one-byte form: always 256 entries (unused ones 0.0)
  for (size_t i = 0; i < all.size(); ++i) std::memcpy(&dict[i + 1], &all[i], sizeof(double));
  return true;
}

// vidx of an already filled SELL layout; dict from value_dictionary (sorted by bit pattern behind dict[0]).  index_bytes = 1: one byte
// per stored entry; 2: two bytes (little endian), for dictionaries beyond 256 entries.
inline void sell_value_index(SellHost& sh, int index_bytes = 1) {
  std::vector<uint64_t> key(sh.dict.size(), 0);
  int nd = 1;
  for (int i = 1; i < (int)sh.dict.size(); ++i) {
    uint64_t b;
    std::memcpy(&b, &sh.dict[i], sizeof(b));
    if (b == 0) break;  // unused tail (a stored +0.0 maps to entry 0)
    key[i] = b;
    nd = i + 1;
  }
  if (index_bytes == 1 && nd > 256) throw std::runtime_error("value dictionary too large for one-byte indices");
  const int64_t stored = (int64_t)sh.val.size();
  sh.vidx.assign(sh.val.size() * (size_t)index_bytes, 0);
#pragma omp parallel for schedule(static)
  for (int64_t k = 0; k < stored; ++k) {
    uint64_t b;
    std::memcpy(&b, &sh.val[k], sizeof(b));
    if (b == 0) continue;
    const auto it = std::lower_bound(key.begin() + 1, key.begin() + nd, b);
    const uint32_t ix = (uint32_t)(it - key.begin());
    if (index_bytes == 1) {
      sh.vidx[k] = (uint8_t)ix;
    } else {
      sh.vidx[2 * k] = (uint8_t)(ix & 0xffu);
      sh.vidx[2 * k + 1] = (uint8_t)(ix >> 8);
    }
  }
}

// interleave = R > 0 (C = 32 R, no sorting): inside every FULL slice position lane * R + k holds row k * 32 + lane of the slice, so
// that a lane's R rows lie 32 apart and the 32 lanes of a warp touch 32 CONSECUTIVE rows at a time (coalesced gathers and
// epilogue accesses); the kernel computes that map arithmetically, `perm` is filled for the host-side checks only.  The last,
// partial slice keeps the identity.
inline void sell_layout(const LocalCsr& m, int C, int sigma, SellHost& out, bool fill_arrays, int interleave = 0) {
  const int64_t nr = m.nrows;
  const int64_t ns = (nr + C - 1) / C;
  out.perm.resize(nr);
  for (int64_t i = 0; i < nr; ++i) out.perm[i] = (int32_t)i;
  out.permuted = false;
  if (interleave > 0) {
    if (C != 32 * interleave || sigma > 1) throw std::runtime_error("interleaved SELL layout: C = 32 R and no sorting");
    for (int64_t sl = 0; (sl + 1) * C <= nr; ++sl)
      for (int lane = 0; lane < 32; ++lane)
        for (int k = 0; k < interleave; ++k) out.perm[sl * C + lane * interleave + k] = (int32_t)(sl * C + k * 32 + lane);
  }
  if (sigma > 1) {
    for (int64_t w0 = 0; w0 < nr; w0 += sigma) {
      const int64_t w1 = std::min<int64_t>(nr, w0 + sigma);
      std::stable_sort(out.perm.begin() + w0, out.perm.begin() + w1,
                       [&](int32_t a, int32_t b) { return (m.ptr[a + 1] - m.ptr[a]) > (m.ptr[b + 1] - m.ptr[b]); });
    }
    for (int64_t i = 0; i < nr && !out.permuted; ++i) out.permuted = out.perm[i] != (int32_t)i;
  }
  out.off.assign(ns + 1, 0);
  for (int64_t sl = 0; sl < ns; ++sl) {
    int64_t w = 0;
    for (int64_t slot = sl * C; slot < std::min<int64_t>(nr, (sl + 1) * C); ++slot) {
      const int32_t r = out.perm[slot];
      w = std::max<int64_t>(w, m.ptr[r + 1] - m.ptr[r]);
    }
    const int64_t nxt = (int64_t)out.off[sl] + w;
    if (nxt * C > INT32_MAX) throw std::runtime_error("SELL storage exceeds int32 entries");
    out.off[sl + 1] = (int32_t)nxt;
  }
  const int64_t stored = (int64_t)out.off[ns] * C;
  out.fill = m.nnz() ? (double)stored / (double)m.nnz() : 1.0;
  if (!fill_arrays) return;
  out.col.assign(stored + 4, 0);
  out.val.assign(stored + 4, 0.0);
#pragma omp parallel for schedule(static)
  for (int64_t sl = 0; sl < ns; ++sl) {
    const int64_t w = out.off[sl + 1] - out.off[sl];
    for (int64_t q = 0; q < C; ++q) {
      const int64_t slot = sl * C + q;
      if (slot >= nr) continue;  // tail rows of the last slice stay (0.0, column 0)
      const int32_t r = out.perm[slot];
      const int64_t b = m.ptr[r], len = m.ptr[r + 1] - b;
      const int32_t padcol = len ? m.col[b + len - 1] : 0;
      for (int64_t j = 0; j < w; ++j) {
        const int64_t dst = ((int64_t)out.off[sl] + j) * C + q;
        out.col[dst] = j < len ? m.col[b + j] : padcol;
        out.val[dst] = j < len ? m.val[b + j] : 0.0;
      }
    }
  }
}

// ---- SELL with implied columns ("diagonal" layout, kernels.cuh k_spmv_sell_diag) -----------------------------
// Stencil operators hold every row's entries at columns row + off[j] for a few fixed offsets.  Slot j of every row then stands
// for column row + off[j], so a slot stores its one value-index byte and no column.  Slices of 128 rows; inside a slice
// ndiag groups of 128 bytes, one per offset (diagonal-major), each with the four-rows-per-lane interleave of the 128-row
// value-indexed layout: byte 4 lane + k is row base + 32 k + lane of a full slice, row base + 4 lane + k of the partial last
// slice.  Code DIAG_ABSENT marks a slot without an entry (rows at the domain boundary, tail rows of the last slice).
// A block qualifies when every row's columns are strictly ascending (then ascending offset = stored order, so the kernel adds
// the products in CSR order), it has at most DIAG_MAX_OFFSETS distinct offsets, ndiag * nrows <= DIAG_MAX_FILL * nnz, and at
// most DIAG_MAX_VALUES distinct non-zero values (value_dictionary's dictionary and order; code 255 stays free).
constexpr int DIAG_MAX_OFFSETS = 32;
constexpr double DIAG_MAX_FILL = 1.25;
constexpr int DIAG_MAX_VALUES = 254;
constexpr uint8_t DIAG_ABSENT = 255;

struct DiagHost {
  std::vector<int32_t> off;  // [ndiag] ascending; empty when the block does not qualify
  std::vector<double> dict;  // [256] (value_dictionary)
  std::vector<uint8_t> idx;  // [nslices * ndiag * 128]
  int64_t nslices = 0;
};

// Returns false (out.off empty) when m does not qualify; fill_arrays = false stops after the checks.
inline bool diag_layout(const LocalCsr& m, DiagHost& out, bool fill_arrays) {
  out = DiagHost();
  const int64_t nr = m.nrows, nnz = m.nnz();
  if (nr <= 0 || m.ncols != nr || m.ptr.empty() || nnz == 0 || nr > INT32_MAX / 2) return false;
  std::vector<int64_t> all;
  bool refused = false;
#pragma omp parallel
  {
    std::vector<int64_t> mine;  // sorted, at most DIAG_MAX_OFFSETS + 1 entries
#pragma omp for schedule(static)
    for (int64_t i = 0; i < nr; ++i) {
      bool stop;
#pragma omp atomic read
      stop = refused;
      if (stop) continue;
      bool ok = true;
      for (int64_t k = m.ptr[i]; k < m.ptr[i + 1] && ok; ++k) {
        if (k > m.ptr[i] && m.col[k] <= m.col[k - 1]) ok = false;
        const int64_t o = (int64_t)m.col[k] - i;
        auto it = std::lower_bound(mine.begin(), mine.end(), o);
        if (it == mine.end() || *it != o) {
          mine.insert(it, o);
          if ((int)mine.size() > DIAG_MAX_OFFSETS) ok = false;
        }
      }
      if (!ok) {
#pragma omp atomic write
        refused = true;
      }
    }
#pragma omp critical
    all.insert(all.end(), mine.begin(), mine.end());
  }
  if (refused) return false;
  std::sort(all.begin(), all.end());
  all.erase(std::unique(all.begin(), all.end()), all.end());
  const int nd = (int)all.size();
  if (nd > DIAG_MAX_OFFSETS || (double)nd * (double)nr > DIAG_MAX_FILL * (double)nnz) return false;
  if (!value_dictionary(m, out.dict, DIAG_MAX_VALUES)) return false;
  out.off.assign(all.begin(), all.end());
  out.nslices = (nr + 127) / 128;
  if (!fill_arrays) return true;
  std::vector<uint64_t> key(1, 0);  // dictionary bit patterns behind dict[0] = +0.0
  for (int i = 1; i < (int)out.dict.size(); ++i) {
    uint64_t b;
    std::memcpy(&b, &out.dict[i], sizeof(b));
    if (b == 0) break;
    key.push_back(b);
  }
  out.idx.assign((size_t)out.nslices * nd * 128, DIAG_ABSENT);
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < nr; ++i) {
    const int64_t sl = i / 128, q = i % 128;
    const int64_t pos = (sl + 1) * 128 <= nr ? (q % 32) * 4 + q / 32 : q;
    int j = 0;
    for (int64_t k = m.ptr[i]; k < m.ptr[i + 1]; ++k) {
      const int64_t o = (int64_t)m.col[k] - i;
      while (out.off[j] != o) ++j;  // both ascending, o is one of the offsets
      uint64_t b;
      std::memcpy(&b, &m.val[k], sizeof(b));
      const uint8_t code = b == 0 ? 0 : (uint8_t)(std::lower_bound(key.begin() + 1, key.end(), b) - key.begin());
      out.idx[(size_t)(sl * nd + j) * 128 + pos] = code;
    }
  }
  return true;
}

// ---- CSR-stream row blocks -----------------------------------------------------------------------------
// Greedy runs of consecutive rows with <= max_rows rows and <= max_entries entries; blk[k] = {first row, first
// entry}, closed by {nrows, nnz}.  Returns false (blk unusable) when a single row exceeds max_entries.
inline bool stream_row_blocks(const LocalCsr& m, int max_rows, int max_entries, std::vector<std::pair<int32_t, int32_t>>& blk) {
  const int64_t nr = m.nrows;
  blk.clear();
  int64_t r = 0;
  while (r < nr) {
    const int64_t e0 = m.ptr[r];
    int64_t r1 = r;
    while (r1 < nr && r1 - r < max_rows && m.ptr[r1 + 1] - e0 <= max_entries) ++r1;
    if (r1 == r) return false;
    blk.emplace_back((int32_t)r, (int32_t)e0);
    r = r1;
  }
  blk.emplace_back((int32_t)nr, (int32_t)(nr ? m.ptr[nr] : 0));
  return true;
}

// ---- boundary rows -------------------------------------------------------------------------------------
// Rows of the own-own block that also have own-ghost entries, stored whole: entries [ptr[k], mid[k]) index the own
// vector, [mid[k], ptr[k+1]) the ghost slots; skip[row] = 1 marks them for the main pass.
struct BndHost {
  std::vector<int32_t> rows, ptr, mid, col;
  std::vector<double> val;
  std::vector<uint8_t> skip;
  int lanes = 1;  // threads per row of the boundary role
};

inline void bnd_layout(const LocalCsr& oo, const LocalCsr& og, BndHost& d) {
  const int64_t nr = oo.nrows;
  d = BndHost();
  d.ptr.push_back(0);
  d.skip.assign((size_t)std::max<int64_t>(nr, 1), 0);
  if (!og.ptr.empty())
    for (int64_t i = 0; i < nr; ++i) {
      if (og.ptr[i + 1] == og.ptr[i]) continue;
      d.rows.push_back((int32_t)i);
      d.skip[i] = 1;
      if (!oo.ptr.empty())
        for (int64_t k = oo.ptr[i]; k < oo.ptr[i + 1]; ++k) {
          d.col.push_back(oo.col[k]);
          d.val.push_back(oo.val[k]);
        }
      d.mid.push_back((int32_t)d.col.size());
      for (int64_t k = og.ptr[i]; k < og.ptr[i + 1]; ++k) {
        d.col.push_back(og.col[k]);
        d.val.push_back(og.val[k]);
      }
      d.ptr.push_back((int32_t)d.col.size());
    }
  // latency-bound role: one thread per row up to 16 entries (all its loads are independent), wider above
  const double mean = d.rows.empty() ? 0.0 : (double)d.col.size() / (double)d.rows.size();
  d.lanes = mean <= 16 ? 1 : mean <= 32 ? 2 : mean <= 64 ? 4 : mean <= 128 ? 8 : mean <= 256 ? 16 : 32;
}

}  // namespace pamg
