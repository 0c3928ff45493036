// Host-side mesh preprocessing (see prep.h).
#include "prep.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <functional>
#include <memory>
#include <numeric>
#include <stdexcept>
#include <string>
#include <thread>

#include <chrono>
#include <cstdio>

namespace shakti {

// SHAKTI_TRACE_PREP=1: wall time of every preprocessing phase on stderr (lap("name") closes a phase)
struct PrepLaps {
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  void operator()(const char* name) {
    static const bool on = getenv("SHAKTI_TRACE_PREP") != nullptr;
    const auto now = std::chrono::steady_clock::now();
    if (on) fprintf(stderr, "[prep] %-32s %8.3f s\n", name, std::chrono::duration<double>(now - t).count());
    t = now;
  }
};

// ------------------------------------------------------------------ host threads
// The preprocessing is embarrassingly parallel over rows / cells / blocks; it runs once per model but on
// 16M-dof meshes one thread needs ~15 s.  SHAKTI_HOST_THREADS overrides the default (hardware threads, at
// most 16, divided among the ranks of a multi-GPU job: they all preprocess at the same time).
static int g_host_thread_share = 1;
static int host_threads() {
  if (const char* e = getenv("SHAKTI_HOST_THREADS")) return std::max(1, atoi(e));
  const int hw = (int)std::thread::hardware_concurrency();
  return std::max(1, std::min(16, hw > 0 ? hw / std::max(1, g_host_thread_share) : 1));
}
// fn(begin, end, thread index) over [0, n) in contiguous chunks
template <class F>
static void parallel_for(int64_t n, F fn, int64_t min_per_thread = 4096) {
  const int nt = (int)std::max<int64_t>(1, std::min<int64_t>(host_threads(), n / std::max<int64_t>(min_per_thread, 1)));
  if (nt <= 1) { fn((int64_t)0, n, 0); return; }
  std::vector<std::thread> th;
  std::vector<std::exception_ptr> err(nt);
  for (int t = 0; t < nt; ++t)
    th.emplace_back([&, t]() {
      try { fn(n * t / nt, n * (t + 1) / nt, t); } catch (...) { err[t] = std::current_exception(); }
    });
  for (auto& x : th) x.join();
  for (auto& e : err)
    if (e) std::rethrow_exception(e);
}
// stable parallel sort: sorted chunks, then pairwise stable merges
template <class It, class Cmp>
static void parallel_stable_sort(It first, It last, Cmp cmp) {
  const int64_t n = last - first;
  int nt = (int)std::max<int64_t>(1, std::min<int64_t>(host_threads(), n / 65536));
  if (nt <= 1) { std::stable_sort(first, last, cmp); return; }
  std::vector<int64_t> cut(nt + 1);
  for (int t = 0; t <= nt; ++t) cut[t] = n * t / nt;
  parallel_for(nt, [&](int64_t a, int64_t b, int) { for (int64_t t = a; t < b; ++t) std::stable_sort(first + cut[t], first + cut[t + 1], cmp); }, 1);
  while (cut.size() > 2) {
    const size_t pairs = (cut.size() - 1) / 2;
    parallel_for((int64_t)pairs, [&](int64_t a, int64_t b, int) {
      for (int64_t k = a; k < b; ++k) std::inplace_merge(first + cut[2 * k], first + cut[2 * k + 1], first + cut[2 * k + 2], cmp);
    }, 1);
    std::vector<int64_t> next;
    for (size_t k = 0; k < cut.size(); k += 2) next.push_back(cut[k]);
    if (next.back() != n) next.push_back(n);
    cut.swap(next);
  }
}

// ------------------------------------------------------------------ generic sparse helpers

HostSell sell_from_csr(const HostCsr& a) {
  HostSell s;
  s.n_rows = a.n_rows;
  s.n_cols = a.n_cols;
  s.n_slices = (a.n_rows + 31) / 32;
  s.slice_ptr.assign(s.n_slices + 1, 0);
  s.rowlen.resize(a.n_rows);
  for (int64_t r = 0; r < a.n_rows; ++r) s.rowlen[r] = a.rowptr[r + 1] - a.rowptr[r];
  int64_t off = 0;
  for (int64_t sl = 0; sl < s.n_slices; ++sl) {
    int w = 0;
    for (int64_t r = sl * 32; r < std::min<int64_t>(a.n_rows, sl * 32 + 32); ++r) w = std::max(w, s.rowlen[r]);
    s.slice_ptr[sl] = (int32_t)off;
    off += 32 * (int64_t)w;
    if (off > 2000000000LL) throw std::runtime_error("SELL matrix too large for int32 offsets");
  }
  s.slice_ptr[s.n_slices] = (int32_t)off;
  s.col.resize(off);
  parallel_for(s.n_slices, [&](int64_t s0, int64_t s1, int) {
    for (int64_t sl = s0; sl < s1; ++sl) {
      int w = (s.slice_ptr[sl + 1] - s.slice_ptr[sl]) / 32;
      for (int lane = 0; lane < 32; ++lane) {
        int64_t r = sl * 32 + lane;
        int32_t padcol = (int32_t)std::min<int64_t>(std::min<int64_t>(r, a.n_rows - 1), a.n_cols - 1);
        if (padcol < 0) padcol = 0;
        for (int k = 0; k < w; ++k) {
          int64_t p = (int64_t)s.slice_ptr[sl] + 32 * (int64_t)k + lane;
          if (r < a.n_rows && k < s.rowlen[r]) s.col[p] = a.col[a.rowptr[r] + k];
          else s.col[p] = padcol;
        }
      }
    }
  }, 256);
  return s;
}

std::vector<int32_t> sell_positions(const HostCsr& a, const HostSell& s) {
  std::vector<int32_t> pos(a.nnz());
  for (int64_t r = 0; r < a.n_rows; ++r)
    for (int32_t k = a.rowptr[r]; k < a.rowptr[r + 1]; ++k) pos[k] = (int32_t)s.pos(r, k - a.rowptr[r]);
  return pos;
}

HostCsr csr_transpose(const HostCsr& a, std::vector<int32_t>* entry_map) {
  HostCsr t;
  t.n_rows = a.n_cols;
  t.n_cols = a.n_rows;
  t.rowptr.assign(t.n_rows + 1, 0);
  for (int32_t c : a.col) t.rowptr[c + 1]++;
  for (int64_t i = 0; i < t.n_rows; ++i) t.rowptr[i + 1] += t.rowptr[i];
  t.col.resize(a.nnz());
  if (entry_map) entry_map->resize(a.nnz());
  std::vector<int32_t> fill(t.rowptr.begin(), t.rowptr.end() - 1);
  for (int64_t r = 0; r < a.n_rows; ++r)
    for (int32_t k = a.rowptr[r]; k < a.rowptr[r + 1]; ++k) {
      int32_t p = fill[a.col[k]]++;
      t.col[p] = (int32_t)r;  // rows visited ascending => columns of t sorted
      if (entry_map) (*entry_map)[p] = k;
    }
  return t;
}

// adjacency (incl. diagonal) of rows [0,n_rows) given cells in some numbering; a row is
// built only if row_of(vertex) >= 0.
struct RawAdj : HostCsr {
  std::unique_ptr<int32_t[]> raw;   // unsorted neighbour lists; rowptr indexes it until finish_rows has run
};
template <class RowOf>
static RawAdj adjacency(int64_t n_rows, int64_t n_cols, int64_t ne, const int32_t* cells, RowOf row_of) {
  // Unsorted neighbour lists (with duplicates) of rows [0, n_rows): every cell contributes the two other
  // vertices to each of its rows, plus one trailing placeholder per row for the diagonal.  Counting and
  // filling run on all host threads with relaxed atomic counters; the order inside a row is therefore
  // arbitrary, which does not matter because finish_rows sorts every row.
  RawAdj a;
  a.n_rows = n_rows;
  a.n_cols = n_cols;
  PrepLaps lap;
  std::vector<int32_t> cnt(n_rows + 1, 0);
  parallel_for(ne, [&](int64_t e0, int64_t e1, int) {
    for (int64_t e = e0; e < e1; ++e)
      for (int i = 0; i < 3; ++i) {
        const int64_t r = row_of(cells[3 * e + i]);
        if (r >= 0) __atomic_fetch_add(&cnt[r + 1], 2, __ATOMIC_RELAXED);
      }
  });
  lap("  adjacency: count");
  std::vector<int64_t> ptr(n_rows + 1, 0);
  for (int64_t r = 0; r < n_rows; ++r) ptr[r + 1] = ptr[r] + cnt[r + 1] + 1;  // + the diagonal
  if (ptr[n_rows] > 2000000000LL) throw std::runtime_error("adjacency too large for int32 offsets");
  // not value-initialised: zero-filling 0.8 GB on one thread (16M dofs) cost more than counting and filling;
  // every element is written below, the pages are first touched by the threads that fill them
  std::unique_ptr<int32_t[]> tmp_own(new int32_t[(size_t)ptr[n_rows]]);
  int32_t* tmp = tmp_own.get();
  std::vector<int64_t> fill(ptr.begin(), ptr.end() - 1);
  lap("  adjacency: alloc");
  parallel_for(ne, [&](int64_t e0, int64_t e1, int) {
    for (int64_t e = e0; e < e1; ++e)
      for (int i = 0; i < 3; ++i) {
        const int64_t r = row_of(cells[3 * e + i]);
        if (r < 0) continue;
        const int64_t p = __atomic_fetch_add(&fill[r], (int64_t)2, __ATOMIC_RELAXED);
        tmp[p] = cells[3 * e + (i + 1) % 3];
        tmp[p + 1] = cells[3 * e + (i + 2) % 3];
      }
  });
  lap("  adjacency: fill");
  // (the last slot of every row is the diagonal's: finish_rows writes its id there)
  a.raw = std::move(tmp_own);
  a.rowptr.resize(n_rows + 1);
  for (int64_t r = 0; r <= n_rows; ++r) a.rowptr[r] = (int32_t)ptr[r];
  return a;
}

// finish: replace the trailing -1 of each row by diag id, sort, unique, compact
static void finish_rows(RawAdj& a, const std::vector<int32_t>& diag_id) {
  const int64_t n = a.n_rows;
  PrepLaps lap;
  std::vector<int32_t> newptr(n + 1, 0), len(n, 0);
  parallel_for(n, [&](int64_t r0, int64_t r1, int) {
    for (int64_t r = r0; r < r1; ++r) {
      int32_t* b = a.raw.get() + a.rowptr[r];
      int32_t* e = a.raw.get() + a.rowptr[r + 1];
      *(e - 1) = diag_id[r];
      std::sort(b, e);
      len[r] = (int32_t)(std::unique(b, e) - b);
    }
  });
  lap("  rows: sort + unique");
  for (int64_t r = 0; r < n; ++r) newptr[r + 1] = newptr[r] + len[r];
  std::vector<int32_t> col(newptr[n]);
  parallel_for(n, [&](int64_t r0, int64_t r1, int) {
    for (int64_t r = r0; r < r1; ++r) std::copy_n(a.raw.get() + a.rowptr[r], len[r], col.data() + newptr[r]);
  });
  a.col.swap(col);
  a.rowptr.swap(newptr);
  a.raw.reset();
  lap("  rows: compact");
}

HostCsr caller_csr(int64_t nv, int64_t ne, const int32_t* cells) {
  RawAdj a = adjacency(nv, nv, ne, cells, [](int32_t v) { return (int64_t)v; });
  std::vector<int32_t> diag(nv);
  std::iota(diag.begin(), diag.end(), 0);
  finish_rows(a, diag);
  return HostCsr(std::move(static_cast<HostCsr&>(a)));
}

std::vector<int32_t> locate_dirichlet_dofs(int64_t nv, int64_t ne, const int32_t* cells,
                                           const uint8_t* marker) {
  // count incident cells per undirected edge (i<j) at the CSR position (i,j)
  HostCsr a = caller_csr(nv, ne, cells);
  std::vector<uint8_t> cnt(a.nnz(), 0);
  auto find = [&](int32_t i, int32_t j) {
    const int32_t* b = a.col.data() + a.rowptr[i];
    const int32_t* e = a.col.data() + a.rowptr[i + 1];
    return (int64_t)(std::lower_bound(b, e, j) - a.col.data());
  };
  for (int64_t c = 0; c < ne; ++c)
    for (int i = 0; i < 3; ++i) {
      int32_t u = cells[3 * c + i], v = cells[3 * c + (i + 1) % 3];
      if (u > v) std::swap(u, v);
      int64_t p = find(u, v);
      if (cnt[p] < 255) cnt[p]++;
    }
  std::vector<uint8_t> is(nv, 0);
  for (int64_t i = 0; i < nv; ++i)
    for (int32_t k = a.rowptr[i]; k < a.rowptr[i + 1]; ++k) {
      int32_t j = a.col[k];
      if (j > i && cnt[k] == 1 && marker[i] && marker[j]) is[i] = is[j] = 1;
    }
  std::vector<int32_t> out;
  for (int64_t i = 0; i < nv; ++i)
    if (is[i]) out.push_back((int32_t)i);
  return out;
}

// ------------------------------------------------------------------ assembly row blocks

void build_assembly_blocks(const HostMesh& m, int32_t max_cells_per_block, AssemblyBlocks& out) {
  const int32_t no = m.n_owned, ne = m.ne;
  PrepLaps lap;
  // vertex -> (cell, local index) incidence of owned rows, cells ascending
  // (counted and filled on all threads with relaxed atomic counters, then every row's short list is sorted:
  // the same arrays as a serial pass over the cells in ascending order)
  std::vector<int32_t> vptr(no + 1, 0);
  parallel_for(ne, [&](int64_t e0, int64_t e1, int) {
    for (int64_t e = e0; e < e1; ++e)
      for (int a = 0; a < 3; ++a) {
        const int32_t r = m.cells[3 * (size_t)e + a];
        if (r < no) __atomic_fetch_add(&vptr[r + 1], 1, __ATOMIC_RELAXED);
      }
  });
  for (int32_t r = 0; r < no; ++r) vptr[r + 1] += vptr[r];
  std::vector<int32_t> vinc(vptr[no]);   // e*4 + a
  {
    std::vector<int32_t> fill(vptr.begin(), vptr.end() - 1);
    parallel_for(ne, [&](int64_t e0, int64_t e1, int) {
      for (int64_t e = e0; e < e1; ++e)
        for (int a = 0; a < 3; ++a) {
          const int32_t r = m.cells[3 * (size_t)e + a];
          if (r < no) vinc[__atomic_fetch_add(&fill[r], 1, __ATOMIC_RELAXED)] = (int32_t)e * 4 + a;
        }
    });
    parallel_for(no, [&](int64_t r0, int64_t r1, int) {
      for (int64_t r = r0; r < r1; ++r) std::sort(vinc.begin() + vptr[r], vinc.begin() + vptr[r + 1]);
    });
  }
  // Blocks are independent: threads take contiguous runs of blocks, collect their variable-length lists
  // locally and the runs are concatenated in block order afterwards (same arrays as a serial pass).
  struct Part {
    std::vector<int32_t> elems, halo, ecount, hcount, rowinc;   // per block: #cells, #halo vertices; per row: #incident cells
    std::vector<uint16_t> lv, inc;
    int32_t max_cells = 0, max_verts = 0;
    bool fits = true, manifold = true;
  };
  lap("assembly plan: incidence");
  for (int32_t rb : {256, 128, 64, 32}) {
    out = AssemblyBlocks();
    out.rows_per_block = rb;
    out.n_blocks = (no + rb - 1) / rb;
    out.src.assign(m.S.padded(), 0xFFFFFFFFu);
    const int nt_max = host_threads();
    std::vector<Part> parts(std::max(1, nt_max));
    int nt_used = 1;
    parallel_for(out.n_blocks, [&](int64_t B0, int64_t B1, int t) {
      Part& P = parts[t];
      std::vector<int32_t> elems, halo;
      for (int64_t B = B0; B < B1 && P.fits; ++B) {
        const int32_t r0 = (int32_t)B * rb, r1 = std::min(no, r0 + rb);
        elems.clear();
        for (int32_t r = r0; r < r1; ++r)
          for (int32_t k = vptr[r]; k < vptr[r + 1]; ++k) elems.push_back(vinc[k] >> 2);
        std::sort(elems.begin(), elems.end());
        elems.erase(std::unique(elems.begin(), elems.end()), elems.end());
        if ((int32_t)elems.size() > max_cells_per_block || elems.size() >= 4096) { P.fits = false; break; }
        auto lidx = [&](int32_t e) { return (int32_t)(std::lower_bound(elems.begin(), elems.end(), e) - elems.begin()); };
        P.max_cells = std::max<int32_t>(P.max_cells, (int32_t)elems.size());
        P.elems.insert(P.elems.end(), elems.begin(), elems.end());
        P.ecount.push_back((int32_t)elems.size());
        // vertices of the block: its own rows first, then the other vertices of its cells (ascending)
        halo.clear();
        for (int32_t e : elems)
          for (int a = 0; a < 3; ++a) {
            const int32_t v = m.cells[3 * (size_t)e + a];
            if (v < r0 || v >= r1) halo.push_back(v);
          }
        std::sort(halo.begin(), halo.end());
        halo.erase(std::unique(halo.begin(), halo.end()), halo.end());
        if ((size_t)(r1 - r0) + halo.size() >= 65535) { P.fits = false; break; }
        P.max_verts = std::max<int32_t>(P.max_verts, (int32_t)((r1 - r0) + halo.size()));
        for (int32_t e : elems)
          for (int a = 0; a < 3; ++a) {
            const int32_t v = m.cells[3 * (size_t)e + a];
            uint16_t lv;
            if (v >= r0 && v < r1) lv = (uint16_t)(v - r0);
            else lv = (uint16_t)((r1 - r0) + (std::lower_bound(halo.begin(), halo.end(), v) - halo.begin()));
            P.lv.push_back(lv);
          }
        P.halo.insert(P.halo.end(), halo.begin(), halo.end());
        P.hcount.push_back((int32_t)halo.size());
        std::vector<int32_t> loc;   // block-local index of each incident cell of the current row
        for (int32_t r = r0; r < r1; ++r) {
          loc.clear();
          for (int32_t k = vptr[r]; k < vptr[r + 1]; ++k) {
            loc.push_back(lidx(vinc[k] >> 2));
            P.inc.push_back((uint16_t)(loc.back() * 4 + (vinc[k] & 3)));
          }
          P.rowinc.push_back(vptr[r + 1] - vptr[r]);
          // Jacobian entries of row r (positions belong to this row alone: written in place)
          for (int32_t kk = m.A.rowptr[r]; kk < m.A.rowptr[r + 1]; ++kk) {
            const int32_t c = m.A.col[kk];
            const int64_t p = m.S.pos(r, kk - m.A.rowptr[r]);
            if (c == r) { out.src[p] = 0xFFFEFFFEu; continue; }
            uint32_t codes[2] = {0xFFFFu, 0xFFFFu};
            int found = 0;
            for (int32_t k = vptr[r]; k < vptr[r + 1]; ++k) {
              const int32_t e = vinc[k] >> 2, a = vinc[k] & 3;
              for (int bb = 0; bb < 3; ++bb)
                if (m.cells[3 * (size_t)e + bb] == c) {
                  if (found < 2) codes[found] = (uint32_t)(loc[k - vptr[r]] * 16 + 3 * a + bb);
                  ++found;
                }
            }
            if (found > 2) P.manifold = false;
            out.src[p] = codes[0] | (codes[1] << 16);
          }
        }
      }
      (void)nt_used;
    }, 8);
    bool fits = true, manifold = true;
    for (const Part& P : parts) { fits &= P.fits; manifold &= P.manifold; }
    lap("assembly plan: blocks");
    if (!fits) continue;
    // concatenate the runs (threads hold ascending, contiguous block ranges): offsets first, then every
    // run is copied to its place by its own thread
    const size_t np = parts.size();
    std::vector<size_t> oe(np + 1, 0), oh(np + 1, 0), oi(np + 1, 0), ob(np + 1, 0), orow(np + 1, 0);
    for (size_t t = 0; t < np; ++t) {
      const Part& P = parts[t];
      out.max_cells = std::max(out.max_cells, P.max_cells);
      out.max_verts = std::max(out.max_verts, P.max_verts);
      oe[t + 1] = oe[t] + P.elems.size();
      oh[t + 1] = oh[t] + P.halo.size();
      oi[t + 1] = oi[t] + P.inc.size();
      ob[t + 1] = ob[t] + P.ecount.size();
      orow[t + 1] = orow[t] + P.rowinc.size();
    }
    out.blk_elems.resize(oe[np]);
    out.blk_lv.resize(3 * oe[np]);
    out.blk_halo.resize(oh[np]);
    out.inc_code.resize(oi[np]);
    out.blk_eptr.assign(ob[np] + 1, 0);
    out.blk_hptr.assign(ob[np] + 1, 0);
    out.inc_ptr.assign(orow[np] + 1, 0);
    parallel_for((int64_t)np, [&](int64_t t0, int64_t t1, int) {
      for (int64_t t = t0; t < t1; ++t) {
        const Part& P = parts[t];
        std::copy(P.elems.begin(), P.elems.end(), out.blk_elems.begin() + oe[t]);
        std::copy(P.lv.begin(), P.lv.end(), out.blk_lv.begin() + 3 * oe[t]);
        std::copy(P.halo.begin(), P.halo.end(), out.blk_halo.begin() + oh[t]);
        std::copy(P.inc.begin(), P.inc.end(), out.inc_code.begin() + oi[t]);
        int32_t acc = (int32_t)oe[t];
        for (size_t k = 0; k < P.ecount.size(); ++k) { acc += P.ecount[k]; out.blk_eptr[ob[t] + k + 1] = acc; }
        acc = (int32_t)oh[t];
        for (size_t k = 0; k < P.hcount.size(); ++k) { acc += P.hcount[k]; out.blk_hptr[ob[t] + k + 1] = acc; }
        acc = (int32_t)oi[t];
        for (size_t k = 0; k < P.rowinc.size(); ++k) { acc += P.rowinc[k]; out.inc_ptr[orow[t] + k + 1] = acc; }
      }
    }, 1);
    out.ok = manifold;
    lap("assembly plan: concatenate");
    return;
  }
  out.ok = false;
}

// ------------------------------------------------------------------ Morton ordering

static inline uint64_t spread_bits(uint64_t v) {  // 21 bits -> every 2nd bit
  v &= 0x1fffff;
  v = (v | (v << 16)) & 0x0000ffff0000ffffULL;
  v = (v | (v << 8)) & 0x00ff00ff00ff00ffULL;
  v = (v | (v << 4)) & 0x0f0f0f0f0f0f0f0fULL;
  v = (v | (v << 2)) & 0x3333333333333333ULL;
  v = (v | (v << 1)) & 0x5555555555555555ULL;
  return v;
}

static std::vector<int32_t> morton_order(int64_t nv, const double* xy) {
  double xmin = 1e300, xmax = -1e300, ymin = 1e300, ymax = -1e300;
  for (int64_t i = 0; i < nv; ++i) {
    xmin = std::min(xmin, xy[2 * i]); xmax = std::max(xmax, xy[2 * i]);
    ymin = std::min(ymin, xy[2 * i + 1]); ymax = std::max(ymax, xy[2 * i + 1]);
  }
  // one common scale so that tiles are square in physical space
  double ext = std::max(xmax - xmin, ymax - ymin);
  if (!(ext > 0)) ext = 1.0;
  const double scale = (double)((1 << 20) - 1) / ext;
  std::vector<std::pair<uint64_t, int32_t>> key(nv);
  parallel_for(nv, [&](int64_t a, int64_t b, int) {
    for (int64_t i = a; i < b; ++i) {
      uint64_t qx = (uint64_t)((xy[2 * i] - xmin) * scale);
      uint64_t qy = (uint64_t)((xy[2 * i + 1] - ymin) * scale);
      key[i] = {spread_bits(qx) | (spread_bits(qy) << 1), (int32_t)i};
    }
  });
  // (key, vertex id) pairs are all distinct, so the order is the same whichever sort produces it
  parallel_stable_sort(key.begin(), key.end(), [](const std::pair<uint64_t, int32_t>& p, const std::pair<uint64_t, int32_t>& q) { return p < q; });
  std::vector<int32_t> order(nv);
  for (int64_t i = 0; i < nv; ++i) order[i] = key[i].second;
  return order;
}

// ------------------------------------------------------------------ the rank-local mesh

void build_host_mesh(int64_t nv, int64_t ne, const double* xy, const int32_t* cells, int rank,
                     int nranks, int reorder, HostMesh& m) {
  if (nv <= 0 || ne <= 0) throw std::runtime_error("empty mesh");
  if (nv > 2000000000LL || ne > 2000000000LL / 3) throw std::runtime_error("mesh too large for int32 indices");
  {
    // Every rank validates the GLOBAL mesh, so that all ranks of a job fail together.  A vertex that belongs to no
    // cell would be an empty Jacobian row (a singular system); DOLFINx never creates such a dof -- its mesh builder
    // keeps only the nodes the cells refer to, and so does meshio_lite.read_msh_arrays -- so it is refused here
    // with a message instead of producing NaNs in the first solve.
    std::vector<uint8_t> used(nv, 0);
    for (int64_t i = 0; i < 3 * ne; ++i) {
      if (cells[i] < 0 || cells[i] >= nv) throw std::runtime_error("cell vertex id out of range");
      used[cells[i]] = 1;
    }
    for (int64_t v = 0; v < nv; ++v)
      if (!used[v])
        throw std::runtime_error("vertex " + std::to_string(v) + " belongs to no cell: remove unreferenced nodes before "
                                 "shakti_create (DOLFINx drops them when it builds the mesh)");
    // non-finite coordinates or a cell of zero area make 1/det J infinite in every kernel: name the cell instead
    int64_t bad_cell = -1;
    parallel_for(ne, [&](int64_t e0, int64_t e1, int) {
      for (int64_t e = e0; e < e1; ++e) {
        const int32_t* c = cells + 3 * e;
        const double d1x = xy[2 * (int64_t)c[1]] - xy[2 * (int64_t)c[0]], d1y = xy[2 * (int64_t)c[1] + 1] - xy[2 * (int64_t)c[0] + 1];
        const double d2x = xy[2 * (int64_t)c[2]] - xy[2 * (int64_t)c[0]], d2y = xy[2 * (int64_t)c[2] + 1] - xy[2 * (int64_t)c[0] + 1];
        const double det = d1x * d2y - d2x * d1y;
        if (!(std::fabs(det) > 0.0) || !std::isfinite(det)) __atomic_store_n(&bad_cell, e, __ATOMIC_RELAXED);
      }
    });
    if (bad_cell >= 0)
      throw std::runtime_error("cell " + std::to_string(bad_cell) + " has zero area or non-finite vertex coordinates");
  }
  m.nv_g = nv; m.ne_g = ne; m.rank = rank; m.nranks = nranks;
  g_host_thread_share = std::max(1, nranks);
  PrepLaps lap;
  std::vector<int32_t> order;
  if (reorder) order = morton_order(nv, xy);
  else { order.resize(nv); std::iota(order.begin(), order.end(), 0); }
  lap("morton order");
  std::vector<int32_t> posof(nv);
  parallel_for(nv, [&](int64_t a, int64_t b, int) { for (int64_t p = a; p < b; ++p) posof[order[p]] = (int32_t)p; });
  std::vector<int64_t> bounds(nranks + 1);
  for (int r = 0; r <= nranks; ++r) bounds[r] = (nv * (int64_t)r) / nranks;
  auto owner_of_pos = [&](int64_t p) {
    return (int)(std::upper_bound(bounds.begin(), bounds.end(), p) - bounds.begin()) - 1;
  };
  const int64_t lo = bounds[rank], hi = bounds[rank + 1];
  m.n_owned = (int32_t)(hi - lo);
  // local cells (any owned vertex) and ghost vertices
  std::vector<int32_t> lc;
  std::vector<int32_t> ghost_pos;
  if (nranks == 1) {
    lc.resize(ne);
    std::iota(lc.begin(), lc.end(), 0);
  } else {
    std::vector<uint8_t> seen(nv, 0);
    for (int64_t e = 0; e < ne; ++e) {
      bool any = false;
      for (int i = 0; i < 3; ++i) {
        int64_t p = posof[cells[3 * e + i]];
        any |= (p >= lo && p < hi);
      }
      if (!any) continue;
      lc.push_back((int32_t)e);
      for (int i = 0; i < 3; ++i) {
        int32_t v = cells[3 * e + i];
        int64_t p = posof[v];
        if ((p < lo || p >= hi) && !seen[v]) { seen[v] = 1; ghost_pos.push_back((int32_t)p); }
      }
    }
    std::sort(ghost_pos.begin(), ghost_pos.end());
  }
  m.n_local = m.n_owned + (int32_t)ghost_pos.size();
  lap("local cells + ghosts");
  m.l2g.resize(m.n_local);
  parallel_for(hi - lo, [&](int64_t a, int64_t b, int) { for (int64_t p = a; p < b; ++p) m.l2g[p] = order[lo + p]; });
  for (size_t k = 0; k < ghost_pos.size(); ++k) m.l2g[m.n_owned + k] = order[ghost_pos[k]];
  m.g2l.assign(nv, -1);
  parallel_for(m.n_local, [&](int64_t a, int64_t b, int) { for (int64_t l = a; l < b; ++l) m.g2l[m.l2g[l]] = (int32_t)l; });
  // cells in local ids, sorted by min local vertex id (stable => ties by caller cell id)
  m.ne = (int32_t)lc.size();
  {
    std::vector<std::pair<int32_t, int32_t>> key(m.ne);
    parallel_for(m.ne, [&](int64_t a, int64_t b, int) {
      for (int64_t k = a; k < b; ++k) {
        const int32_t* c = cells + 3 * (int64_t)lc[k];
        key[k] = {std::min(m.g2l[c[0]], std::min(m.g2l[c[1]], m.g2l[c[2]])), lc[k]};
      }
    });
    if (reorder) parallel_stable_sort(key.begin(), key.end(), [](const std::pair<int32_t, int32_t>& a, const std::pair<int32_t, int32_t>& b) { return a.first < b.first; });
    m.cell_l2g.resize(m.ne);
    m.cells.resize(3 * (size_t)m.ne);
    parallel_for(m.ne, [&](int64_t a, int64_t b, int) {
      for (int64_t k = a; k < b; ++k) {
        m.cell_l2g[k] = key[k].second;
        const int32_t* c = cells + 3 * (int64_t)key[k].second;
        for (int i = 0; i < 3; ++i) m.cells[3 * (size_t)k + i] = m.g2l[c[i]];
      }
    });
  }
  m.x.resize(m.n_local);
  m.y.resize(m.n_local);
  parallel_for(m.n_local, [&](int64_t a, int64_t b, int) {
    for (int64_t l = a; l < b; ++l) { m.x[l] = xy[2 * (int64_t)m.l2g[l]]; m.y[l] = xy[2 * (int64_t)m.l2g[l] + 1]; }
  });
  lap("maps, cell sort, coordinates");
  // CSR of owned rows
  const int32_t no = m.n_owned;
  {
    RawAdj adj = adjacency(no, m.n_local, m.ne, m.cells.data(), [no](int32_t v) { return v < no ? (int64_t)v : (int64_t)-1; });
    std::vector<int32_t> diag(no);
    std::iota(diag.begin(), diag.end(), 0);
    finish_rows(adj, diag);
    m.A = std::move(static_cast<HostCsr&>(adj));
  }
  m.S = sell_from_csr(m.A);
  lap("CSR + SELL pattern");
  // slot table and diagonal positions
  m.slot.assign(9 * (size_t)m.ne, -1);
  auto find = [&](int32_t r, int32_t c) -> int32_t {
    const int32_t* b = m.A.col.data() + m.A.rowptr[r];
    const int32_t* e = m.A.col.data() + m.A.rowptr[r + 1];
    const int32_t* p = std::lower_bound(b, e, c);
    return (int32_t)m.S.pos(r, (int)(p - b));
  };
  parallel_for(m.ne, [&](int64_t e0, int64_t e1, int) {
    for (int64_t e = e0; e < e1; ++e)
      for (int a = 0; a < 3; ++a) {
        int32_t r = m.cells[3 * (size_t)e + a];
        if (r >= no) continue;
        for (int b = 0; b < 3; ++b) m.slot[(size_t)(3 * a + b) * m.ne + e] = find(r, m.cells[3 * (size_t)e + b]);
      }
  });
  m.diag_pos.resize(no);
  parallel_for(no, [&](int64_t r0, int64_t r1, int) {
    for (int64_t r = r0; r < r1; ++r) m.diag_pos[r] = find((int32_t)r, (int32_t)r);
  });
  lap("slot table + diagonal");
  // winning cell: highest caller cell id containing the vertex
  // (caller cell id << 32 | local cell id), maximised per row with a compare-and-swap loop on all threads:
  // caller ids are distinct, so the maximum -- and with it the result -- does not depend on the visiting order
  m.win_cell.assign(no, -1);
  std::vector<int64_t> win_key(no, -1);
  parallel_for(m.ne, [&](int64_t e0, int64_t e1, int) {
    for (int64_t e = e0; e < e1; ++e)
      for (int a = 0; a < 3; ++a) {
        const int32_t r = m.cells[3 * (size_t)e + a];
        if (r >= no) continue;
        const int64_t k = ((int64_t)m.cell_l2g[e] << 32) | (int64_t)e;
        int64_t cur = __atomic_load_n(&win_key[r], __ATOMIC_RELAXED);
        while (k > cur && !__atomic_compare_exchange_n(&win_key[r], &cur, k, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
      }
  });
  m.win.assign(4 * (size_t)no, 0);
  parallel_for(no, [&](int64_t ra, int64_t rb, int) {
  for (int64_t r = ra; r < rb; ++r) {
    const int32_t e = win_key[r] < 0 ? -1 : (int32_t)(win_key[r] & 0xFFFFFFFFLL);
    if (e >= 0) m.win_cell[r] = m.cell_l2g[e];
    if (e < 0) {  // isolated vertex: degenerate 'cell' of itself (gradients vanish)
      m.win[4 * (size_t)r] = m.win[4 * (size_t)r + 1] = m.win[4 * (size_t)r + 2] = r;
      m.win[4 * (size_t)r + 3] = -1;
      continue;
    }
    int loc = 0;
    for (int a = 0; a < 3; ++a) {
      m.win[4 * (size_t)r + a] = m.cells[3 * (size_t)e + a];
      if (m.cells[3 * (size_t)e + a] == r) loc = a;
    }
    m.win[4 * (size_t)r + 3] = loc;
  }
  });
  lap("winning cells");
  m.cell_counted.assign(m.ne, 1);
  if (nranks > 1)
    parallel_for(m.ne, [&](int64_t e0, int64_t e1, int) {
      for (int64_t e = e0; e < e1; ++e) {
        const int32_t* c = m.cells.data() + 3 * (size_t)e;
        const int32_t g = std::min(m.l2g[c[0]], std::min(m.l2g[c[1]], m.l2g[c[2]]));
        m.cell_counted[e] = owner_of_pos(posof[g]) == rank ? 1 : 0;
      }
    });
  // halo maps
  m.nbrs.clear();
  if (nranks > 1) {
    std::vector<std::vector<int32_t>> send(nranks);
    for (int32_t e = 0; e < m.ne; ++e) {
      int own[3];
      for (int a = 0; a < 3; ++a) own[a] = owner_of_pos(posof[m.l2g[m.cells[3 * (size_t)e + a]]]);
      for (int a = 0; a < 3; ++a) {
        if (own[a] != rank) continue;
        for (int b = 0; b < 3; ++b)
          if (own[b] != rank) send[own[b]].push_back(m.cells[3 * (size_t)e + a]);
      }
    }
    std::vector<int32_t> rb(nranks, 0), rc(nranks, 0);
    for (int32_t g = no; g < m.n_local; ++g) {
      int o = owner_of_pos(posof[m.l2g[g]]);
      if (rc[o] == 0) rb[o] = g;
      rc[o]++;
    }
    for (int r = 0; r < nranks; ++r) {
      auto& s = send[r];
      std::sort(s.begin(), s.end());
      s.erase(std::unique(s.begin(), s.end()), s.end());
      if (s.empty() && rc[r] == 0) continue;
      Neighbor nb;
      nb.rank = r;
      nb.send_local = s;
      nb.recv_begin = rb[r];
      nb.recv_count = rc[r];
      m.nbrs.push_back(std::move(nb));
    }
  }
}

}  // namespace shakti
