// Device data layout shared by every kernel of libamg1d.
//
// Operator storage ("element tiles").  The host uploads each level in the element-block (BSR-like)
// form the C ABI documents; on the device the same numbers are kept interleaved in tiles of
// TILE = 32 consecutive elements:
//
//      mat[tile][k][lane]      tile = e / 32, lane = e % 32, k in [0, K)
//
// so a warp that owns one tile streams one contiguous K*256-byte range and every warp-level load is
// a fully used, 256-byte coalesced request - for ANY block size m, with no shared-memory transpose
// and no bank conflicts.
//
// Which entries k enumerates depends on the level's *structure class*, detected at upload from the
// blocks themselves (amg1d_set_level / amg1d_set_level_pattern scan every off-diagonal block):
//
//   ST_DENSE   (0)  A_lo (m*m), A_di (m*m), A_up (m*m), Dinv          K = 3 m^2 + |Dinv|
//   ST_COLROW  (1)  A_lo has ONE non-zero column `ilo`, A_up ONE non-zero row `iup` - every level the
//                   reference assembles from DG fluxes (src/dg_mesh.jl:181-338: an element sees only
//                   the trace node of its left neighbour, and only its own trace row sees the right
//                   neighbour).  Stored: that column (m), A_di (m*m), that row (m), Dinv.
//                   K = m^2 + 2 m + |Dinv|
//   ST_ROWCOL  (2)  A_lo has ONE non-zero row `ilo`, A_up ONE non-zero column `iup` - CG levels in
//                   the [vertex_k, interior nodes of element k] grouping (only the vertex row couples
//                   to the previous group, and everything couples only to the next group's vertex).
//                   Stored: that row (m), A_di, that column (m), Dinv.      K = m^2 + 2 m + |Dinv|
//   ST_REPEAT  (3)  every column of A_lo is the same vector c, every row of A_up the same vector r (bit for
//                   bit) - the agglomerated pAgg = 1 levels below a DG p = 1 level: that level couples to its
//                   neighbours through one trace node, and every agglomeration transfer maps the trace node's
//                   value to exactly 1.0 in both coarse basis functions, so each Galerkin column / row is the
//                   fine one times 1.0 plus exact zeros.  Stored: c = column 0 of A_lo (m), A_di, r = row 0
//                   of A_up (m), Dinv - the tile rows of ST_COLROW with ilo = iup = 0.
//                   K = m^2 + 2 m + |Dinv|.  Chosen only for block-Jacobi 2 x 2 levels uploaded as
//                   patterns (amg1d_set_level_pattern; amg1d.cu: repeat_eligible says why).
//
// Dropping structural zeros does not change a single bit of the results: fma(0, x, y) == y, and the
// surviving terms are accumulated in the same ascending-column order as the dense form.  ST_REPEAT keeps
// every term of the dense form: the dense chain y[i] = fma(A_lo(i, j), xl[j], y[i]) over ascending j reads
// A_lo(i, j) == c[i] (A_up(i, j) == r[j]), so the same FMAs run on the same operand values.  |Dinv| is
// m*m for a block smoother and m for a diagonal (point-Jacobi) one.  Inside a block the dense parts
// are column-major, k = j*m + i.
//
// Vectors (x, b, r) stay element-major, v[e*m + i], exactly the reference's DG numbering
// (src/dg_mesh.jl:41-46), with ghost elements on each side of the slab: v[-g*m .. -1] and
// v[n*m .. (n+g)*m - 1] exist and hold zeros on a single GPU (A_lo[0] = A_up[n-1] = 0 there) or the
// neighbour rank's edge elements in the sharded case.
#pragma once
#include <cstdint>

#define AMG1D_TILE 32

enum { AMG1D_ST_DENSE = 0, AMG1D_ST_COLROW = 1, AMG1D_ST_ROWCOL = 2, AMG1D_ST_REPEAT = 3 };

struct MatDesc {
    int m, diag, st;
    int ilo, iup;              // see the structure classes above (0 for ST_DENSE and ST_REPEAT)
    int K, o_di, o_up, o_dv;   // tile rows: [0, o_di) A_lo part, [o_di, o_up) A_di, [o_up, o_dv) A_up part, [o_dv, K) Dinv
};

__host__ __device__ inline MatDesc amg1d_desc(int m, int diag, int st, int ilo, int iup) {
    MatDesc d;
    d.m = m; d.diag = diag ? 1 : 0; d.st = st;
    d.ilo = (st == AMG1D_ST_COLROW || st == AMG1D_ST_ROWCOL) ? ilo : 0;
    d.iup = (st == AMG1D_ST_COLROW || st == AMG1D_ST_ROWCOL) ? iup : 0;
    const int off = st ? m : m * m;
    d.o_di = off;
    d.o_up = off + m * m;
    d.o_dv = d.o_up + off;
    d.K = d.o_dv + (diag ? m : m * m);
    return d;
}

// Source of tile row k: which = 0 A_lo, 1 A_di, 2 A_up, 3 Dinv; idx = position inside the uploaded
// block (column-major j*m + i) or inside the Dinv array of the element.
__host__ __device__ inline void amg1d_row_source(const MatDesc& d, int k, int* which, int* idx) {
    const int m = d.m;
    if (k < d.o_di) {
        *which = 0;
        *idx = d.st == AMG1D_ST_DENSE ? k : (d.st == AMG1D_ST_ROWCOL ? k * m + d.ilo : d.ilo * m + k);
    } else if (k < d.o_up) {
        *which = 1;
        *idx = k - d.o_di;
    } else if (k < d.o_dv) {
        const int kk = k - d.o_up;
        *which = 2;
        *idx = d.st == AMG1D_ST_DENSE ? kk : (d.st == AMG1D_ST_ROWCOL ? d.iup * m + kk : kk * m + d.iup);
    } else {
        *which = 3;
        *idx = k - d.o_dv;
    }
}

__host__ __device__ inline int64_t amg1d_tiles(int64_t n) { return (n + AMG1D_TILE - 1) / AMG1D_TILE; }
