// Host-side one-time preprocessing of the mesh: internal (Morton) ordering, partition into
// owned + ghost vertices, owner-computes element overlap, CSR/SELL patterns, winning cells.
// Replaces what DOLFINx does at functionspace / form-compilation time (reference
// source/model_setup.py:29-30, source/solvers.py:51) and its mesh partitioner
// (setups/setup_cooke2.py:19).
#pragma once
#include <cstdint>
#include <vector>

namespace shakti {

// CSR pattern on the host (rows x cols), sorted unique columns per row.
struct HostCsr {
  int64_t n_rows = 0, n_cols = 0;
  std::vector<int32_t> rowptr;  // n_rows + 1
  std::vector<int32_t> col;
  int64_t nnz() const { return (int64_t)col.size(); }
};

// SELL-32 layout derived from a CSR pattern: slice s holds rows [32 s, 32 s + 32), entry k of
// row r sits at slice_ptr[s] + 32 k + (r & 31).  Padding entries point at the row itself
// (column = min(r, n_cols-1)) with value 0.
struct HostSell {
  int64_t n_rows = 0, n_cols = 0, n_slices = 0;
  std::vector<int32_t> slice_ptr;  // n_slices + 1 (entry offsets)
  std::vector<int32_t> col;        // padded
  std::vector<int32_t> rowlen;     // n_rows
  int64_t padded() const { return (int64_t)col.size(); }
  // position of entry k of row r
  inline int64_t pos(int64_t r, int k) const { return (int64_t)slice_ptr[r >> 5] + 32 * (int64_t)k + (r & 31); }
};

HostSell sell_from_csr(const HostCsr& a);
// position map csr entry -> sell entry
std::vector<int32_t> sell_positions(const HostCsr& a, const HostSell& s);
HostCsr csr_transpose(const HostCsr& a, std::vector<int32_t>* entry_map /* t-entry -> a-entry */);

struct Neighbor {
  int rank;
  std::vector<int32_t> send_local;  // owned local ids whose values this rank sends
  int32_t recv_begin, recv_count;   // ghost range [recv_begin, recv_begin+recv_count) (local ids)
};

struct HostMesh {
  int64_t nv_g = 0, ne_g = 0;
  int rank = 0, nranks = 1;
  int32_t n_owned = 0, n_local = 0, ne = 0;
  std::vector<int32_t> l2g;       // local vertex -> caller id (owned first, internal order; then ghosts)
  std::vector<int32_t> g2l;       // caller id -> local id or -1
  std::vector<int32_t> cell_l2g;  // local cell -> caller cell id
  std::vector<int32_t> cells;     // ne x 3 local vertex ids, cell's own vertex order kept
  std::vector<double> x, y;       // n_local
  HostCsr A;                      // owned rows x local cols, columns sorted by local id
  HostSell S;                     // SELL of A
  std::vector<int32_t> slot;      // 9 x ne (k-major: slot[k*ne + e]); SELL position or -1
  std::vector<int32_t> diag_pos;  // n_owned: SELL position of the diagonal
  std::vector<int32_t> win;       // 4 x n_owned: v0,v1,v2 (local ids) of the winning cell, local index
  std::vector<int32_t> win_cell;  // n_owned: caller cell id of the winning cell
  // ne: 1 if this rank counts the cell in global integrals (it owns the cell's vertex with the smallest caller
  // id), else 0 -- every cell is counted on exactly one rank although local cells overlap between ranks
  std::vector<int32_t> cell_counted;
  std::vector<Neighbor> nbrs;
};

// Row-block plan of the atomics-free assembly: a CUDA block owns `rows_per_block` consecutive
// owned rows, computes every cell touching them into shared memory (cells on block borders are
// computed by each block that needs them) and then GATHERS: each row sums its incident cells'
// residual entries, each Jacobian entry the (at most two) cells containing its edge.
struct AssemblyBlocks {
  int32_t rows_per_block = 0, n_blocks = 0, max_cells = 0;
  bool ok = false;                  // false: mesh not edge-manifold -> use the atomic kernel
  int32_t max_verts = 0;            // most vertices (owned rows + halo) any block touches
  std::vector<int32_t> blk_eptr;    // n_blocks + 1
  std::vector<int32_t> blk_elems;   // local cell ids, ascending inside a block
  std::vector<uint16_t> blk_lv;     // 3 per block cell: block-local vertex index (row - r0, or rows_in_block + halo position)
  std::vector<int32_t> blk_hptr;    // n_blocks + 1: halo vertex lists
  std::vector<int32_t> blk_halo;    // local vertex ids outside the block's own rows, ascending
  std::vector<int32_t> inc_ptr;     // n_owned + 1
  std::vector<uint16_t> inc_code;   // (cell index in block) * 4 + local vertex index
  std::vector<uint32_t> src;        // per padded SELL entry: two 16-bit codes (cell index in block)*16 + 3a+b;
                                    // 0xFFFF = none; diagonal entries hold 0xFFFEFFFE (use the incident list)
};
void build_assembly_blocks(const HostMesh& m, int32_t max_cells_per_block, AssemblyBlocks& out);

// Build the rank-local mesh.  `reorder` = 1: Morton ordering of vertices; 0: caller order.
void build_host_mesh(int64_t nv, int64_t ne, const double* xy, const int32_t* cells, int rank,
                     int nranks, int reorder, HostMesh& out);

// CSR pattern in caller numbering (sorted unique columns, diagonal included).
HostCsr caller_csr(int64_t nv, int64_t ne, const int32_t* cells);

// Dofs of boundary facets whose vertices all carry marker != 0 (sorted, caller numbering).
std::vector<int32_t> locate_dirichlet_dofs(int64_t nv, int64_t ne, const int32_t* cells,
                                           const uint8_t* marker);

}  // namespace shakti
