// K8: point-cloud evaluation (the DTU protocol: accuracy / completeness), DESIGN §4 "K8 point-cloud evaluation".
//
// Uniform grid over a cloud of m points.  Fine cells of edge `cell` are grouped into coarse blocks of 8 x 8 x 8 cells, and the
// cell key is block-major: key = block * 512 + (lz * 8 + ly) * 8 + lx with block = (bz * nby + by) * nbx + bx.  Sorting the
// points by key (a stable torch sort) therefore makes every fine cell AND every coarse block one contiguous range.
//
//   pc_grid_keys_kernel      one thread per point: fp64 cell coordinates, clamped to the grid -> int32 key
//   pc_grid_cells_kernel     one thread per sorted position: the point as float4 (x, y, z, original index), and the first / last
//                            point of its cell and of its block -> cells[key] = {begin, end}, blocks[block] = {begin, end}.
//                            Each entry is written by exactly one thread; untouched entries stay {0, 0} (empty).
//   pc_nearest_kernel        one thread per query: exact nearest distance, capped at max_dist (below)
//   pc_thin_count_kernel     thinning (greedy minimum-distance, reducePts_haa) on a grid with cell >= dst: per point the number
//   pc_thin_list_kernel      of lower-ranked points within dst (fp64, inclusive), then the list itself (CSR, scan order)
//   pc_thin_round_kernel     one parallel greedy round: undecided -> kept when every lower-ranked neighbour is removed, removed
//                            when one is kept; reads one state buffer and writes the other, counts the undecided points
//
// Nearest search.  Shells r = 0, 1, ... of fine cells around the query's (clamped) cell, up to kFineShells; then shells of coarse
// blocks, skipping empty blocks, visiting an occupied block by its points (few) or by its fine cells (many).  A shell is entered
// only while a lower bound on the distance to every cell of it and beyond is below min(best, max_dist), so the result is exact:
// a minimum does not depend on the visiting order.  Lower bounds subtract `slack` (set by the host above the fp32 rounding of
// the box coordinates), so a point whose cell was decided in fp64 is never pruned by a rounding of its cell's faces.
#include "common.cuh"

using namespace mvsb200;

namespace {

constexpr int kThreads = 256;
constexpr int kFineShells = 2;      // fine-cell shells before the coarse level takes over (5 x 5 x 5 cells)
constexpr int kDirect = 48;         // an occupied block with at most this many points is scanned point by point
#define kInf __int_as_float(0x7f800000)

struct Grid {
    float ox, oy, oz, cell;
    int nbx, nby, nbz;              // coarse blocks per axis; fine cells per axis = 8 * nb
    double inv;                     // 1 / cell, rounded once on the host
};

__device__ __forceinline__ int key_of(int ix, int iy, int iz, const Grid& g) {
    return ((((iz >> 3) * g.nby + (iy >> 3)) * g.nbx + (ix >> 3)) << 9) | ((iz & 7) << 6) | ((iy & 7) << 3) | (ix & 7);
}

// fp64 product with the host's reciprocal: no division, hence no slow-path call frame in the kernels
__device__ __forceinline__ int cell_of(float x, float o, double inv, int n) {
    const double t = floor(((double)x - (double)o) * inv);
    return (int)fmin(fmax(t, 0.0), (double)(n - 1));
}

// distance along one axis from q to the slab [o + j c, o + (j + 1) c]
__device__ __forceinline__ float gap(float q, float o, float c, int j) {
    const float lo = fmaf((float)j, c, o);
    return fmaxf(fmaxf(lo - q, q - (lo + c)), 0.f);
}

// lower bound on the distance from q to any cell at Chebyshev distance >= r from cell (cx, cy, cz) of a grid of n cells per axis
// with edge c; +inf when no such cell exists
__device__ __forceinline__ float shell_bound(float qx, float qy, float qz, int cx, int cy, int cz, int r, int nx, int ny, int nz,
                                             const Grid& g, float c, float slack) {
    float L = kInf;
    if (cx - r >= 0) L = fminf(L, gap(qx, g.ox, c, cx - r));
    if (cx + r < nx) L = fminf(L, gap(qx, g.ox, c, cx + r));
    if (cy - r >= 0) L = fminf(L, gap(qy, g.oy, c, cy - r));
    if (cy + r < ny) L = fminf(L, gap(qy, g.oy, c, cy + r));
    if (cz - r >= 0) L = fminf(L, gap(qz, g.oz, c, cz - r));
    if (cz + r < nz) L = fminf(L, gap(qz, g.oz, c, cz + r));
    return fmaxf(L - slack, 0.f);
}

__device__ __forceinline__ float sq(float a) { return a * a; }

__device__ __forceinline__ void scan_points(const float4* __restrict__ pts, int b, int e, float qx, float qy, float qz, float& best) {
    for (int p = b; p < e; ++p) {
        const float4 t = __ldg(pts + p);
        best = fminf(best, sq(t.x - qx) + sq(t.y - qy) + sq(t.z - qz));
    }
}

__global__ void __launch_bounds__(kThreads) pc_grid_keys_kernel(const float* __restrict__ xyz, int n, Grid g, int32_t* __restrict__ keys) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int ix = cell_of(xyz[3 * (size_t)i], g.ox, g.inv, 8 * g.nbx);
    const int iy = cell_of(xyz[3 * (size_t)i + 1], g.oy, g.inv, 8 * g.nby);
    const int iz = cell_of(xyz[3 * (size_t)i + 2], g.oz, g.inv, 8 * g.nbz);
    keys[i] = key_of(ix, iy, iz, g);
}

__global__ void __launch_bounds__(kThreads) pc_grid_cells_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ skeys,
                                                                const int64_t* __restrict__ perm, int n, float4* __restrict__ pts,
                                                                int2* __restrict__ cells, int2* __restrict__ blocks) {
    const int s = blockIdx.x * kThreads + threadIdx.x;
    if (s >= n) return;
    const int i = (int)perm[s];
    pts[s] = make_float4(xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], __int_as_float(i));
    const int k = skeys[s];
    const int kp = s > 0 ? skeys[s - 1] : -1, kn = s + 1 < n ? skeys[s + 1] : -1;
    if (k != kp) cells[k].x = s;
    if (k != kn) cells[k].y = s + 1;
    if (kp < 0 || (k >> 9) != (kp >> 9)) blocks[k >> 9].x = s;
    if (kn < 0 || (k >> 9) != (kn >> 9)) blocks[k >> 9].y = s + 1;
}

__global__ void __launch_bounds__(kThreads, 2) pc_nearest_kernel(const float* __restrict__ query, int n, const float4* __restrict__ pts,
                                                             const int2* __restrict__ cells, const int2* __restrict__ blocks, Grid g,
                                                             float slack, float max_dist, float* __restrict__ dist) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const float qx = query[3 * (size_t)i], qy = query[3 * (size_t)i + 1], qz = query[3 * (size_t)i + 2];
    const int nx = 8 * g.nbx, ny = 8 * g.nby, nz = 8 * g.nbz;
    // the grid's box is farther than max_dist: nothing to find (fp64, once per query)
    {
        const double c = g.cell;
        const double ex = fmax(fmax((double)g.ox - qx, (double)qx - (g.ox + nx * c)), 0.0);
        const double ey = fmax(fmax((double)g.oy - qy, (double)qy - (g.oy + ny * c)), 0.0);
        const double ez = fmax(fmax((double)g.oz - qz, (double)qz - (g.oz + nz * c)), 0.0);
        if (ex * ex + ey * ey + ez * ez >= (double)max_dist * max_dist) {
            dist[i] = kInf;
            return;
        }
    }
    const float sl = slack + 2.4e-7f * (fabsf(qx) + fabsf(qy) + fabsf(qz));
    const float lim = max_dist * max_dist;
    const int cx = cell_of(qx, g.ox, g.inv, nx), cy = cell_of(qy, g.oy, g.inv, ny), cz = cell_of(qz, g.oz, g.inv, nz);
    float best = kInf;                                                  // squared
    int r = 0;
    for (; r <= kFineShells; ++r) {
        const float L = shell_bound(qx, qy, qz, cx, cy, cz, r, nx, ny, nz, g, g.cell, sl);
        if (L * L >= fminf(best, lim)) break;
        for (int dz = -r; dz <= r; ++dz) {
            const int iz = cz + dz;
            if (iz < 0 || iz >= nz) continue;
            const float gz = sq(fmaxf(gap(qz, g.oz, g.cell, iz) - sl, 0.f));
            for (int dy = -r; dy <= r; ++dy) {
                const int iy = cy + dy;
                if (iy < 0 || iy >= ny) continue;
                const float gy = gz + sq(fmaxf(gap(qy, g.oy, g.cell, iy) - sl, 0.f));
                const int step = (dz == -r || dz == r || dy == -r || dy == r) ? 1 : max(2 * r, 1);
                for (int dx = -r; dx <= r; dx += step) {
                    const int ix = cx + dx;
                    if (ix < 0 || ix >= nx) continue;
                    if (gy + sq(fmaxf(gap(qx, g.ox, g.cell, ix) - sl, 0.f)) >= fminf(best, lim)) continue;
                    const int2 c = __ldg(cells + key_of(ix, iy, iz, g));
                    scan_points(pts, c.x, c.y, qx, qy, qz, best);
                }
            }
        }
    }
    if (r > kFineShells &&
        sq(shell_bound(qx, qy, qz, cx, cy, cz, kFineShells + 1, nx, ny, nz, g, g.cell, sl)) < fminf(best, lim)) {
        // coarse level: blocks of 8 fine cells per axis; the fine cells within kFineShells of (cx, cy, cz) are done
        const float bc = 8.f * g.cell;
        const int bx = cx >> 3, by = cy >> 3, bz = cz >> 3;
        for (int R = 0;; ++R) {
            const float L = shell_bound(qx, qy, qz, bx, by, bz, R, g.nbx, g.nby, g.nbz, g, bc, sl);
            if (L * L >= fminf(best, lim)) break;
            for (int dz = -R; dz <= R; ++dz) {
                const int jz = bz + dz;
                if (jz < 0 || jz >= g.nbz) continue;
                const float gz = sq(fmaxf(gap(qz, g.oz, bc, jz) - sl, 0.f));
                for (int dy = -R; dy <= R; ++dy) {
                    const int jy = by + dy;
                    if (jy < 0 || jy >= g.nby) continue;
                    const float gy = gz + sq(fmaxf(gap(qy, g.oy, bc, jy) - sl, 0.f));
                    const int step = (dz == -R || dz == R || dy == -R || dy == R) ? 1 : max(2 * R, 1);
                    for (int dx = -R; dx <= R; dx += step) {
                        const int jx = bx + dx;
                        if (jx < 0 || jx >= g.nbx) continue;
                        if (gy + sq(fmaxf(gap(qx, g.ox, bc, jx) - sl, 0.f)) >= fminf(best, lim)) continue;
                        const int blk = (jz * g.nby + jy) * g.nbx + jx;
                        const int2 br = __ldg(blocks + blk);
                        if (br.y <= br.x) continue;                     // empty block
                        if (br.y - br.x <= kDirect) {
                            scan_points(pts, br.x, br.y, qx, qy, qz, best);
                            continue;
                        }
                        for (int lz = 0; lz < 8; ++lz) {
                            const int iz = 8 * jz + lz;
                            const float fz = sq(fmaxf(gap(qz, g.oz, g.cell, iz) - sl, 0.f));
                            if (fz >= fminf(best, lim)) continue;
                            for (int ly = 0; ly < 8; ++ly) {
                                const int iy = 8 * jy + ly;
                                const float fy = fz + sq(fmaxf(gap(qy, g.oy, g.cell, iy) - sl, 0.f));
                                if (fy >= fminf(best, lim)) continue;
                                const bool near_zy = abs(iz - cz) <= kFineShells && abs(iy - cy) <= kFineShells;
                                for (int lx = 0; lx < 8; ++lx) {
                                    const int ix = 8 * jx + lx;
                                    if (near_zy && abs(ix - cx) <= kFineShells) continue;      // visited in the fine shells
                                    if (fy + sq(fmaxf(gap(qx, g.ox, g.cell, ix) - sl, 0.f)) >= fminf(best, lim)) continue;
                                    const int2 c = __ldg(cells + (blk << 9) + (lz << 6) + (ly << 3) + lx);
                                    scan_points(pts, c.x, c.y, qx, qy, qz, best);
                                }
                            }
                        }
                    }
                }
            }
        }
    }
    // sqrt by one Newton step on the approximate reciprocal root (within an ulp; no IEEE slow-path call frame)
    float d = kInf;
    if (best == 0.f) {
        d = 0.f;
    } else if (best < lim) {
        const float y = rsqrtf(best);
        d = best * y;
        d = fmaf(0.5f * y, fmaf(-d, d, best), d);
    }
    dist[i] = d < max_dist ? d : kInf;
}

// the lower-ranked points within dst of sorted point s (fp64 on the fp32 coordinates, inclusive), in scan order; list == NULL: count
__device__ __forceinline__ int thin_neighbours(int s, const float4* __restrict__ pts, const int2* __restrict__ cells,
                                               const int32_t* __restrict__ rank, const Grid& g, double dst2, int32_t* list) {
    const float4 p = pts[s];
    const int rs = rank[s];
    const int nx = 8 * g.nbx, ny = 8 * g.nby, nz = 8 * g.nbz;
    const int cx = cell_of(p.x, g.ox, g.inv, nx), cy = cell_of(p.y, g.oy, g.inv, ny), cz = cell_of(p.z, g.oz, g.inv, nz);
    const float dst2f = (float)dst2 * 1.0001f;
    int cnt = 0;
    for (int iz = max(cz - 1, 0); iz <= min(cz + 1, nz - 1); ++iz)
        for (int iy = max(cy - 1, 0); iy <= min(cy + 1, ny - 1); ++iy)
            for (int ix = max(cx - 1, 0); ix <= min(cx + 1, nx - 1); ++ix) {
                const int2 c = __ldg(cells + key_of(ix, iy, iz, g));
                for (int t = c.x; t < c.y; ++t) {
                    const float4 o = __ldg(pts + t);
                    // fp32 filter well outside its rounding, then the fp64 test of the definition
                    if (sq(o.x - p.x) + sq(o.y - p.y) + sq(o.z - p.z) > dst2f) continue;
                    const double dx = (double)o.x - p.x, dy = (double)o.y - p.y, dz = (double)o.z - p.z;
                    if (dx * dx + dy * dy + dz * dz <= dst2 && __ldg(rank + t) < rs) {
                        if (list) list[cnt] = t;
                        ++cnt;
                    }
                }
            }
    return cnt;
}

__global__ void __launch_bounds__(kThreads, 4) pc_thin_count_kernel(const float4* __restrict__ pts, const int2* __restrict__ cells,
                                                                const int32_t* __restrict__ rank, int n, Grid g, double dst2,
                                                                int32_t* __restrict__ counts) {
    const int s = blockIdx.x * kThreads + threadIdx.x;
    if (s < n) counts[s] = thin_neighbours(s, pts, cells, rank, g, dst2, nullptr);
}

__global__ void __launch_bounds__(kThreads, 4) pc_thin_list_kernel(const float4* __restrict__ pts, const int2* __restrict__ cells,
                                                               const int32_t* __restrict__ rank, int n, Grid g, double dst2,
                                                               const int64_t* __restrict__ offsets, int32_t* __restrict__ list) {
    const int s = blockIdx.x * kThreads + threadIdx.x;
    if (s < n) thin_neighbours(s, pts, cells, rank, g, dst2, list + offsets[s]);
}

// states: 0 undecided, 1 kept, 2 removed
__global__ void __launch_bounds__(kThreads) pc_thin_round_kernel(const int64_t* __restrict__ offsets, const int32_t* __restrict__ list,
                                                                const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int n,
                                                                int32_t* __restrict__ undecided) {
    const int s = blockIdx.x * kThreads + threadIdx.x;
    bool open = false;
    if (s < n) {
        uint8_t st = in[s];
        if (st == 0) {
            bool all_removed = true, any_kept = false;
            for (int64_t k = offsets[s], e = offsets[s + 1]; k < e; ++k) {
                const uint8_t t = in[list[k]];
                if (t == 1) {
                    any_kept = true;
                    break;
                }
                all_removed &= t == 2;
            }
            st = any_kept ? 2 : all_removed ? 1 : 0;
            open = st == 0;
        }
        out[s] = st;
    }
    const int c = __syncthreads_count(open);
    if (threadIdx.x == 0 && c) atomicAdd(undecided, c);         // an integer count: the same total in any order
}

int blocks_for(int n) { return (n + kThreads - 1) / kThreads; }

bool grid_ok(float cell, int nbx, int nby, int nbz) {
    return cell > 0.f && isfinite(cell) && nbx >= 1 && nby >= 1 && nbz >= 1 &&
           (long long)nbx * nby * nbz * 512 <= (long long)MVSB200_PC_MAX_CELLS;
}

}  // namespace

extern "C" int mvsb200_pc_grid_keys(const float* xyz, int n, float ox, float oy, float oz, float cell, int nbx, int nby, int nbz,
                                    int32_t* keys, void* stream) {
    MVS_REQUIRE(xyz && keys, "pc_grid_keys: null pointer");
    MVS_REQUIRE(n >= 1, "pc_grid_keys: 1 <= n < 2^31 points");
    MVS_REQUIRE(grid_ok(cell, nbx, nby, nbz), "pc_grid_keys: cell > 0 and at most %d cells", MVSB200_PC_MAX_CELLS);
    pc_grid_keys_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(xyz, n, Grid{ox, oy, oz, cell, nbx, nby, nbz, 1.0 / (double)cell}, keys);
    MVS_CHECK_LAUNCH("pc_grid_keys");
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_grid_cells(const float* xyz, const int32_t* sorted_keys, const int64_t* perm, int n, float* pts,
                                     int32_t* cells, int32_t* blocks, void* stream) {
    MVS_REQUIRE(xyz && sorted_keys && perm && pts && cells && blocks, "pc_grid_cells: null pointer");
    MVS_REQUIRE(aligned16(pts) && ((uintptr_t)cells & 7) == 0 && ((uintptr_t)blocks & 7) == 0, "pc_grid_cells: misaligned buffer");
    MVS_REQUIRE(n >= 1, "pc_grid_cells: 1 <= n < 2^31 points");
    pc_grid_cells_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(xyz, sorted_keys, perm, n, (float4*)pts, (int2*)cells,
                                                                               (int2*)blocks);
    MVS_CHECK_LAUNCH("pc_grid_cells");
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_nearest(const float* query, int n, const float* pts, const int32_t* cells, const int32_t* blocks, float ox,
                                  float oy, float oz, float cell, int nbx, int nby, int nbz, float slack, float max_dist, float* dist,
                                  void* stream) {
    MVS_REQUIRE(query && pts && cells && blocks && dist, "pc_nearest: null pointer");
    MVS_REQUIRE(aligned16(pts) && ((uintptr_t)cells & 7) == 0 && ((uintptr_t)blocks & 7) == 0, "pc_nearest: misaligned buffer");
    MVS_REQUIRE(n >= 0, "pc_nearest: 0 <= n < 2^31 queries");
    MVS_REQUIRE(grid_ok(cell, nbx, nby, nbz), "pc_nearest: cell > 0 and at most %d cells", MVSB200_PC_MAX_CELLS);
    MVS_REQUIRE(max_dist > 0.f && isfinite(max_dist) && slack >= 0.f, "pc_nearest: max_dist > 0 (finite), slack >= 0");
    if (n == 0) return MVSB200_OK;
    pc_nearest_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(query, n, (const float4*)pts, (const int2*)cells,
                                                                            (const int2*)blocks, Grid{ox, oy, oz, cell, nbx, nby, nbz, 1.0 / (double)cell},
                                                                            slack, max_dist, dist);
    MVS_CHECK_LAUNCH("pc_nearest");
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_thin_neighbours(const float* pts, const int32_t* cells, const int32_t* rank_sorted, int n, float ox, float oy,
                                          float oz, float cell, int nbx, int nby, int nbz, double dst, const int64_t* offsets,
                                          int32_t* counts, int32_t* list, void* stream) {
    MVS_REQUIRE(pts && cells && rank_sorted, "pc_thin_neighbours: null pointer");
    MVS_REQUIRE(offsets ? list != nullptr : counts != nullptr, "pc_thin_neighbours: counts, or offsets and list");
    MVS_REQUIRE(aligned16(pts) && ((uintptr_t)cells & 7) == 0, "pc_thin_neighbours: misaligned buffer");
    MVS_REQUIRE(n >= 1, "pc_thin_neighbours: 1 <= n < 2^31 points");
    MVS_REQUIRE(grid_ok(cell, nbx, nby, nbz), "pc_thin_neighbours: cell > 0 and at most %d cells", MVSB200_PC_MAX_CELLS);
    MVS_REQUIRE(dst > 0.0 && (double)cell >= dst, "pc_thin_neighbours: 0 < dst <= cell");
    const Grid g{ox, oy, oz, cell, nbx, nby, nbz, 1.0 / (double)cell};
    if (offsets) {
        pc_thin_list_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>((const float4*)pts, (const int2*)cells, rank_sorted, n, g,
                                                                                  dst * dst, offsets, list);
        MVS_CHECK_LAUNCH("pc_thin_list");
    } else {
        pc_thin_count_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>((const float4*)pts, (const int2*)cells, rank_sorted, n, g,
                                                                                   dst * dst, counts);
        MVS_CHECK_LAUNCH("pc_thin_count");
    }
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_thin_round(const int64_t* offsets, const int32_t* list, const uint8_t* state_in, uint8_t* state_out, int n,
                                     int32_t* undecided, void* stream) {
    MVS_REQUIRE(offsets && list && state_in && state_out && undecided, "pc_thin_round: null pointer");
    MVS_REQUIRE(state_in != state_out, "pc_thin_round: the state buffers must differ");
    MVS_REQUIRE(n >= 1, "pc_thin_round: 1 <= n < 2^31 points");
    pc_thin_round_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(offsets, list, state_in, state_out, n, undecided);
    MVS_CHECK_LAUNCH("pc_thin_round");
    return MVSB200_OK;
}
