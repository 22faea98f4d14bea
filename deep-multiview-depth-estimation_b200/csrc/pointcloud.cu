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
//   pc_nearest_kernel        one thread per query: exact nearest distance, capped at max_dist (below); <true>: and its index
//   pc_thin_count_kernel     thinning (greedy minimum-distance, reducePts_haa) on a grid with cell >= dst: per point the number
//   pc_thin_list_kernel      of lower-ranked points within dst (fp64, inclusive), then the list itself (CSR, scan order)
//   pc_thin_round_kernel     one parallel greedy round: undecided -> kept when every lower-ranked neighbour is removed, removed
//                            when one is kept; reads one state buffer and writes the other, counts the undecided points
//   pc_transform_crop_kernel K9, Tanks and Temples: fp64 affine transform and polygon-volume crop, one thread per point
//   pc_voxel_keys_kernel     K9: int64 voxel key of each fp64 point
//   pc_voxel_mean_kernel     K9: one thread per occupied voxel, the sequential fp64 mean of its stably sorted points
//   pc_icp_sums_{a,b}_kernel K9 registration: the Umeyama sums of the correspondences in two passes, a deterministic fp64 reduction
//   pc_transform64_kernel    K9 registration: an fp64 affine update of the source in place, and its fp32 rounding
//   pc_knn_kernel            K10: one thread per query, the exact k nearest points in the order (d^2, index), capped at max_dist;
//                            <true>: on the cloud itself, the normal of each point's neighbourhood (fp64 covariance, Jacobi)
//
// Grid search (grid_search, the one traversal of pc_nearest_kernel and pc_knn_kernel).  Shells r = 0, 1, ... of fine cells around
// the query's (clamped) cell, up to kFineShells; then shells of coarse blocks, skipping empty blocks, visiting an occupied block by
// its points (few) or by its fine cells (many).  A shell is entered, and a cell or block visited, only while a lower bound on its
// distance is below the caller's squared bound: min(best, max_dist^2) for the nearest point, the k-th entry of the list for the k
// nearest.  So every point below the bound is visited and the result is exact: neither a minimum nor a list in a total order
// depends on the visiting order.  Lower bounds subtract `slack` (set by the host above the fp32 rounding of the box coordinates),
// so a point whose cell was decided in fp64 is never pruned by a rounding of its cell's faces, and a point that ties the bound is
// never pruned.  The one variation: the k-nearest list must not hold a point twice, so there a sparse block within one block of
// the query's (it may hold fine cells the shells visited) is visited by its fine cells rather than point by point.
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

// IDX: also the original index of the best point (pts[].w), the smaller index on an exact tie of the squared fp32 distance
template <bool IDX>
__device__ __forceinline__ void scan_points(const float4* __restrict__ pts, int b, int e, float qx, float qy, float qz, float& best,
                                            int& bi) {
    for (int p = b; p < e; ++p) {
        const float4 t = __ldg(pts + p);
        const float d = sq(t.x - qx) + sq(t.y - qy) + sq(t.z - qz);
        if constexpr (IDX) {
            const int j = __float_as_int(t.w);
            if (d < best || (d == best && j < bi)) best = d, bi = j;
        } else {
            best = fminf(best, d);
        }
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

// the squared distance from q to the grid's box of nx x ny x nz fine cells (fp64, once per query)
__device__ __forceinline__ double box_gap2(float qx, float qy, float qz, const Grid& g, int nx, int ny, int nz) {
    const double c = g.cell;
    const double ex = fmax(fmax((double)g.ox - qx, (double)qx - (g.ox + nx * c)), 0.0);
    const double ey = fmax(fmax((double)g.oy - qy, (double)qy - (g.oy + ny * c)), 0.0);
    const double ez = fmax(fmax((double)g.oz - qz, (double)qz - (g.oz + nz * c)), 0.0);
    return ex * ex + ey * ey + ez * ez;
}

// the square root of s by one Newton step on the approximate reciprocal root (within an ulp; no IEEE slow-path call frame),
// +inf for s >= lim
__device__ __forceinline__ float root_below(float s, float lim) {
    float d = kInf;
    if (s == 0.f) {
        d = 0.f;
    } else if (s < lim) {
        const float y = rsqrtf(s);
        d = s * y;
        d = fmaf(0.5f * y, fmaf(-d, d, s), d);
    }
    return d;
}

// The search of the header comment around query q in its cell (cx, cy, cz), with `sl` the query's slack.  bound(): the current
// squared pruning bound, compared with every lower bound (a point at the bound is not pruned: the bounds lie sl below the true
// gaps); scan(b, e): visit the sorted points [b, e).  ONCE: every point is visited at most once, so a sparse block within one block
// of the query's is visited by its fine cells; without it such a block is scanned point by point, and a point of the fine shells
// may be visited again, which a minimum does not notice.
template <bool ONCE, class Bound, class Scan>
__device__ __forceinline__ void grid_search(float qx, float qy, float qz, int cx, int cy, int cz, const Grid& g, float sl,
                                            const int2* __restrict__ cells, const int2* __restrict__ blocks, Bound bound, Scan scan) {
    const int nx = 8 * g.nbx, ny = 8 * g.nby, nz = 8 * g.nbz;
    int r = 0;
    for (; r <= kFineShells; ++r) {
        const float L = shell_bound(qx, qy, qz, cx, cy, cz, r, nx, ny, nz, g, g.cell, sl);
        if (L * L >= bound()) break;
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
                    if (gy + sq(fmaxf(gap(qx, g.ox, g.cell, ix) - sl, 0.f)) >= bound()) continue;
                    const int2 c = __ldg(cells + key_of(ix, iy, iz, g));
                    scan(c.x, c.y);
                }
            }
        }
    }
    if (r > kFineShells && sq(shell_bound(qx, qy, qz, cx, cy, cz, kFineShells + 1, nx, ny, nz, g, g.cell, sl)) < bound()) {
        // coarse level: blocks of 8 fine cells per axis; the fine cells within kFineShells of (cx, cy, cz) are done
        const float bc = 8.f * g.cell;
        const int bx = cx >> 3, by = cy >> 3, bz = cz >> 3;
        for (int R = 0;; ++R) {
            const float L = shell_bound(qx, qy, qz, bx, by, bz, R, g.nbx, g.nby, g.nbz, g, bc, sl);
            if (L * L >= bound()) break;
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
                        if (gy + sq(fmaxf(gap(qx, g.ox, bc, jx) - sl, 0.f)) >= bound()) continue;
                        const int blk = (jz * g.nby + jy) * g.nbx + jx;
                        const int2 br = __ldg(blocks + blk);
                        if (br.y <= br.x) continue;                     // empty block
                        if (br.y - br.x <= kDirect && (!ONCE || R > 1)) {
                            scan(br.x, br.y);
                            continue;
                        }
                        for (int lz = 0; lz < 8; ++lz) {
                            const int iz = 8 * jz + lz;
                            const float fz = sq(fmaxf(gap(qz, g.oz, g.cell, iz) - sl, 0.f));
                            if (fz >= bound()) continue;
                            for (int ly = 0; ly < 8; ++ly) {
                                const int iy = 8 * jy + ly;
                                const float fy = fz + sq(fmaxf(gap(qy, g.oy, g.cell, iy) - sl, 0.f));
                                if (fy >= bound()) continue;
                                const bool near_zy = abs(iz - cz) <= kFineShells && abs(iy - cy) <= kFineShells;
                                for (int lx = 0; lx < 8; ++lx) {
                                    const int ix = 8 * jx + lx;
                                    if (near_zy && abs(ix - cx) <= kFineShells) continue;      // visited in the fine shells
                                    if (fy + sq(fmaxf(gap(qx, g.ox, g.cell, ix) - sl, 0.f)) >= bound()) continue;
                                    const int2 c = __ldg(cells + (blk << 9) + (lz << 6) + (ly << 3) + lx);
                                    scan(c.x, c.y);
                                }
                            }
                        }
                    }
                }
            }
        }
    }
}

// IDX: also index[i] = the original index of the nearest point (ties: the smaller index), -1 where dist[i] is +inf
template <bool IDX>
__global__ void __launch_bounds__(kThreads, 2) pc_nearest_kernel(const float* __restrict__ query, int n, const float4* __restrict__ pts,
                                                             const int2* __restrict__ cells, const int2* __restrict__ blocks, Grid g,
                                                             float slack, float max_dist, float* __restrict__ dist,
                                                             int32_t* __restrict__ index) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const float qx = query[3 * (size_t)i], qy = query[3 * (size_t)i + 1], qz = query[3 * (size_t)i + 2];
    const int nx = 8 * g.nbx, ny = 8 * g.nby, nz = 8 * g.nbz;
    if (box_gap2(qx, qy, qz, g, nx, ny, nz) >= (double)max_dist * max_dist) {          // nothing within max_dist
        dist[i] = kInf;
        if constexpr (IDX) index[i] = -1;
        return;
    }
    const float sl = slack + 2.4e-7f * (fabsf(qx) + fabsf(qy) + fabsf(qz));
    const float lim = max_dist * max_dist;
    const int cx = cell_of(qx, g.ox, g.inv, nx), cy = cell_of(qy, g.oy, g.inv, ny), cz = cell_of(qz, g.oz, g.inv, nz);
    float best = kInf;                                                  // squared
    int bi = -1;
    grid_search<false>(qx, qy, qz, cx, cy, cz, g, sl, cells, blocks, [&] { return fminf(best, lim); },
                       [&](int b, int e) { scan_points<IDX>(pts, b, e, qx, qy, qz, best, bi); });
    const float d = root_below(best, lim);
    dist[i] = d < max_dist ? d : kInf;
    if constexpr (IDX) index[i] = d < max_dist ? bi : -1;
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

// ---- Tanks and Temples pre-processing (DESIGN §4 "K9 Tanks and Temples evaluation") -------------------------------------------
// fp64 with explicit round-to-nearest intrinsics, so that nvcc contracts nothing into an FMA: every bit equals a numpy restatement
// written in the same operation order.

constexpr int kMaxPolygon = 1024;

struct Affine {
    double a[12];                   // rows 0..2 of a 4 x 4 matrix whose last row is (0, 0, 0, 1), row-major
};

// one thread per point: p' = A [p; 1] (skipped when `transform` is 0), then Open3D's SelectionPolygonVolume::CropInPolygon with the
// polygon's (u, v) columns in shared memory: outside when p_w is outside [axis_min, axis_max]; else inside iff an odd number of the
// edge nodes crossing p_v lie below p_u
__global__ void __launch_bounds__(kThreads) pc_transform_crop_kernel(const float* __restrict__ xyz, int n, Affine A, int transform,
                                                                    const double* __restrict__ polygon, int k, int u, int v, int w,
                                                                    double axis_min, double axis_max, double* __restrict__ out,
                                                                    uint8_t* __restrict__ keep) {
    __shared__ double bu[kMaxPolygon], bv[kMaxPolygon];
    for (int t = threadIdx.x; t < k; t += kThreads) {
        bu[t] = polygon[3 * t + u];
        bv[t] = polygon[3 * t + v];
    }
    __syncthreads();
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    double p[3] = {xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2]};
    if (transform) {
        double q[3];
#pragma unroll
        for (int r = 0; r < 3; ++r)
            q[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(A.a[4 * r], p[0]), __dmul_rn(A.a[4 * r + 1], p[1])),
                                       __dmul_rn(A.a[4 * r + 2], p[2])), A.a[4 * r + 3]);
        p[0] = q[0], p[1] = q[1], p[2] = q[2];
    }
    out[3 * (size_t)i] = p[0], out[3 * (size_t)i + 1] = p[1], out[3 * (size_t)i + 2] = p[2];
    // selects, not p[u]: a run-time index would put p in a local-memory stack frame
    const double pu = u == 0 ? p[0] : p[1], pv = v == 1 ? p[1] : p[2], pw = w == 0 ? p[0] : w == 1 ? p[1] : p[2];
    bool in = false;
    if (!(pw < axis_min || pw > axis_max)) {
        for (int a = 0; a < k; ++a) {
            const int b = a + 1 == k ? 0 : a + 1;
            const double av = bv[a], bvv = bv[b];
            if ((av < pv && bvv >= pv) || (bvv < pv && av >= pv)) {
                const double node = __dadd_rn(bu[a], __dmul_rn(__ddiv_rn(__dsub_rn(pv, av), __dsub_rn(bvv, av)), __dsub_rn(bu[b], bu[a])));
                in ^= node < pu;
            }
        }
    }
    keep[i] = in;
}

// one thread per point: the voxel index floor((p - vmin) / voxel) per axis (IEEE division) -> int64 key (iz ny + iy) nx + ix
__global__ void __launch_bounds__(kThreads) pc_voxel_keys_kernel(const double* __restrict__ xyz, int n, double ox, double oy, double oz,
                                                                double voxel, int64_t nx, int64_t ny, int64_t* __restrict__ keys) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int64_t ix = (int64_t)floor(__ddiv_rn(__dsub_rn(xyz[3 * (size_t)i], ox), voxel));
    const int64_t iy = (int64_t)floor(__ddiv_rn(__dsub_rn(xyz[3 * (size_t)i + 1], oy), voxel));
    const int64_t iz = (int64_t)floor(__ddiv_rn(__dsub_rn(xyz[3 * (size_t)i + 2], oz), voxel));
    keys[i] = (iz * ny + iy) * nx + ix;
}

// one thread per occupied voxel: its points are perm[offsets[j] .. offsets[j + 1]) (a stable sort: ascending input order), summed
// one after another from 0 in fp64, then divided by their count
__global__ void __launch_bounds__(kThreads) pc_voxel_mean_kernel(const double* __restrict__ xyz, const int64_t* __restrict__ perm,
                                                                const int64_t* __restrict__ offsets, int n_voxels,
                                                                double* __restrict__ mean, float* __restrict__ mean_f32) {
    const int j = blockIdx.x * kThreads + threadIdx.x;
    if (j >= n_voxels) return;
    const int64_t b = offsets[j], e = offsets[j + 1];
    double sx = 0.0, sy = 0.0, sz = 0.0;
    for (int64_t s = b; s < e; ++s) {
        const int64_t i = __ldg(perm + s);
        sx = __dadd_rn(sx, __ldg(xyz + 3 * i));
        sy = __dadd_rn(sy, __ldg(xyz + 3 * i + 1));
        sz = __dadd_rn(sz, __ldg(xyz + 3 * i + 2));
    }
    const double c = (double)(e - b);
    const double m[3] = {__ddiv_rn(sx, c), __ddiv_rn(sy, c), __ddiv_rn(sz, c)};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        mean[3 * (size_t)j + r] = m[r];
        mean_f32[3 * (size_t)j + r] = (float)m[r];
    }
}

// ---- K9 registration: the ICP loop of the toolbox's three stages (DESIGN §4 "K9 registration") ------------------------------------
// Per correspondence i -> index[i] (>= 0) of the source src [n, 3] fp64 and the target tgt [m, 3] fp64, two passes, each a fixed
// grid-stride split over at most kSumBlocks blocks, a fixed shared-memory tree per block, per-block fp64 partials, and the last block
// to finish (an integer ticket) adding the partials in block order with the same tree.  No float atomics: the bits depend on n only.
//   pass A  sums[0..7]  = c, sum |s - t|^2, sum s (3), sum t (3)
//   pass B  sums[8..17] = sum (t - mu_t)(s - mu_s)^T (row-major, t's axis first), sum |s - mu_s|^2, with mu = sum / c read from
//           pass A's sums in device memory (zeros when c = 0)

constexpr int kSumBlocks = MVSB200_PC_ICP_BLOCKS;
constexpr int kSumsA = 8, kSumsB = 10;

// the block's K values -> partial[blockIdx.x]; the last block adds the partials in block order -> out[0..K); its ticket is reset
template <int K>
__device__ __forceinline__ void reduce_sums(double (&v)[K], double* __restrict__ partial, double* __restrict__ out,
                                            unsigned* __restrict__ ticket) {
    __shared__ double sh[K][kThreads];
    __shared__ bool last;
    const int t = threadIdx.x;
#pragma unroll
    for (int k = 0; k < K; ++k) sh[k][t] = v[k];
    __syncthreads();
    for (int h = kThreads / 2; h > 0; h >>= 1) {
        if (t < h) {
#pragma unroll
            for (int k = 0; k < K; ++k) sh[k][t] = __dadd_rn(sh[k][t], sh[k][t + h]);
        }
        __syncthreads();
    }
    if (t < K) partial[(size_t)blockIdx.x * K + t] = sh[t][0];
    __threadfence();
    __syncthreads();
    if (t == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double a = 0.0;
        for (int b = t; b < (int)gridDim.x; b += kThreads) a = __dadd_rn(a, __ldcg(partial + (size_t)b * K + k));
        sh[k][t] = a;
    }
    __syncthreads();
    for (int h = kThreads / 2; h > 0; h >>= 1) {
        if (t < h) {
#pragma unroll
            for (int k = 0; k < K; ++k) sh[k][t] = __dadd_rn(sh[k][t], sh[k][t + h]);
        }
        __syncthreads();
    }
    if (t < K) out[t] = sh[t][0];
    if (t == 0) *ticket = 0u;
}

__global__ void __launch_bounds__(kThreads) pc_icp_sums_a_kernel(const double* __restrict__ src, const int32_t* __restrict__ index, int n,
                                                                const double* __restrict__ tgt, double* __restrict__ partial,
                                                                double* __restrict__ sums, unsigned* __restrict__ ticket) {
    double v[kSumsA] = {};
    for (int i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
        const int j = __ldg(index + i);
        if (j < 0) continue;
        const double sx = __ldg(src + 3 * (size_t)i), sy = __ldg(src + 3 * (size_t)i + 1), sz = __ldg(src + 3 * (size_t)i + 2);
        const double tx = __ldg(tgt + 3 * (size_t)j), ty = __ldg(tgt + 3 * (size_t)j + 1), tz = __ldg(tgt + 3 * (size_t)j + 2);
        const double dx = sx - tx, dy = sy - ty, dz = sz - tz;
        v[0] += 1.0;
        v[1] += dx * dx + dy * dy + dz * dz;
        v[2] += sx, v[3] += sy, v[4] += sz;
        v[5] += tx, v[6] += ty, v[7] += tz;
    }
    reduce_sums<kSumsA>(v, partial, sums, ticket);
}

__global__ void __launch_bounds__(kThreads) pc_icp_sums_b_kernel(const double* __restrict__ src, const int32_t* __restrict__ index, int n,
                                                                const double* __restrict__ tgt, double* __restrict__ partial,
                                                                double* __restrict__ sums, unsigned* __restrict__ ticket) {
    const double c = sums[0];
    double ms[3] = {0.0, 0.0, 0.0}, mt[3] = {0.0, 0.0, 0.0};
    if (c > 0.0) {
#pragma unroll
        for (int r = 0; r < 3; ++r) ms[r] = __ddiv_rn(sums[2 + r], c), mt[r] = __ddiv_rn(sums[5 + r], c);
    }
    double v[kSumsB] = {};
    for (int i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
        const int j = __ldg(index + i);
        if (j < 0) continue;
        double a[3], b[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) a[r] = __ldg(src + 3 * (size_t)i + r) - ms[r], b[r] = __ldg(tgt + 3 * (size_t)j + r) - mt[r];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int q = 0; q < 3; ++q) v[3 * r + q] += b[r] * a[q];
        v[9] += a[0] * a[0] + a[1] * a[1] + a[2] * a[2];
    }
    reduce_sums<kSumsB>(v, partial, sums + kSumsA, ticket);
}

// one thread per point, in place: p' = A [p; 1] in K9's operation order (no contraction), and its fp32 rounding
__global__ void __launch_bounds__(kThreads) pc_transform64_kernel(double* __restrict__ xyz, int n, Affine A, float* __restrict__ xyz_f32) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const double p[3] = {xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2]};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const double q = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(A.a[4 * r], p[0]), __dmul_rn(A.a[4 * r + 1], p[1])),
                                             __dmul_rn(A.a[4 * r + 2], p[2])), A.a[4 * r + 3]);
        xyz[3 * (size_t)i + r] = q;
        xyz_f32[3 * (size_t)i + r] = (float)q;
    }
}

// ---- K9 trajectory alignment: the toolbox's RANSAC over camera centres (DESIGN §4 "K9 trajectory alignment") --------------------
// Correspondences i <-> i of src [n, 3] (the camera centres to register) and tgt [n, 3] (the reference centres), fp64.
//   pc_ransac_hyp_kernel     one thread per hypothesis h: its ransac_n counter-based draws, Eigen's Umeyama on them with a
//                            one-sided Jacobi SVD, then good / error2 over every correspondence, staged through shared memory in
//                            tiles that every thread of the block reads at the same address
//   pc_ransac_select_kernel  one block: the lexicographic best (max good, min rmse, min h) in a fixed strided scan and a fixed tree;
//                            the comparison is a total order, so the winner does not depend on the split

constexpr int kHypThreads = 128;
constexpr int kAlignTile = 256;
constexpr int kSelectThreads = 256;
constexpr int kJacobiSweeps = 16;
constexpr int kMaxSample = MVSB200_PC_RANSAC_MAX_SAMPLE;

// draw j of hypothesis h: a SplitMix64 step from seed at counter h * ransac_n + j + 1, reduced mod n
__device__ __forceinline__ int ransac_draw(uint64_t seed, int h, int ransac_n, int j, int n) {
    uint64_t z = seed + ((uint64_t)h * (uint64_t)ransac_n + (uint64_t)j + 1ull) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return (int)((z ^ (z >> 31)) % (uint64_t)n);
}

// one Jacobi rotation of columns P, Q of B = Sigma V (b[column][row]) that makes them orthogonal; V accumulates it
template <int P, int Q>
__device__ __forceinline__ bool jacobi_pair(double (&b)[3][3], double (&v)[3][3]) {
    const double alpha = b[P][0] * b[P][0] + b[P][1] * b[P][1] + b[P][2] * b[P][2];
    const double beta = b[Q][0] * b[Q][0] + b[Q][1] * b[Q][1] + b[Q][2] * b[Q][2];
    const double gamma = b[P][0] * b[Q][0] + b[P][1] * b[Q][1] + b[P][2] * b[Q][2];
    if (!(fabs(gamma) > 1e-15 * sqrt(alpha * beta))) return false;
    const double zeta = (beta - alpha) / (2.0 * gamma);
    const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
    const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const double bp = b[P][r], bq = b[Q][r], vp = v[P][r], vq = v[Q][r];
        b[P][r] = c * bp - s * bq, b[Q][r] = s * bp + c * bq;
        v[P][r] = c * vp - s * vq, v[Q][r] = s * vp + c * vq;
    }
    return true;
}

// Eigen's umeyama(src^T, dst^T, with_scaling) on the pairs drawn for hypothesis h -> T, rows 0..2 of [cR | t].  False (T
// untouched) when the draws hold fewer than 3 distinct indices.  Sigma = (1/k) sum (t - mu_t)(s - mu_s)^T = B V^T after the
// sweeps, with V a product of rotations (det V = +1); for the column k of smallest norm and (i, j, k) a cyclic order,
// u_i = b_i / |b_i|, u_j = b_j / |b_j| and w = u_i x u_j give R = U S V^T = u_i v_i^T + u_j v_j^T + w v_k^T and
// tr(D S) = |b_i| + |b_j| + b_k . w, whichever sign the third left singular vector takes.
__device__ __forceinline__ bool ransac_umeyama(const double* __restrict__ src, const double* __restrict__ tgt, int n, uint64_t seed,
                                               int h, int rn, int with_scaling, double (&T)[12]) {
    const int a = ransac_draw(seed, h, rn, 0, n);
    int b2 = -1;
    bool three = false;
    for (int j = 1; j < rn; ++j) {
        const int i = ransac_draw(seed, h, rn, j, n);
        if (i != a) {
            if (b2 < 0) b2 = i;
            else three |= i != b2;
        }
    }
    if (!three) return false;
    const double inv = 1.0 / (double)rn;
    double ms[3] = {0.0, 0.0, 0.0}, mt[3] = {0.0, 0.0, 0.0};
    for (int j = 0; j < rn; ++j) {
        const size_t i = (size_t)ransac_draw(seed, h, rn, j, n);
#pragma unroll
        for (int r = 0; r < 3; ++r) ms[r] += __ldg(src + 3 * i + r), mt[r] += __ldg(tgt + 3 * i + r);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) ms[r] *= inv, mt[r] *= inv;
    double b[3][3] = {}, var = 0.0;                 // b[q][r] = Sigma[r][q]: column q
    for (int j = 0; j < rn; ++j) {
        const size_t i = (size_t)ransac_draw(seed, h, rn, j, n);
        double ds[3], dt[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) ds[r] = __ldg(src + 3 * i + r) - ms[r], dt[r] = __ldg(tgt + 3 * i + r) - mt[r];
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
            for (int r = 0; r < 3; ++r) b[q][r] += dt[r] * ds[q];
        var += ds[0] * ds[0] + ds[1] * ds[1] + ds[2] * ds[2];
    }
#pragma unroll
    for (int q = 0; q < 3; ++q)
#pragma unroll
        for (int r = 0; r < 3; ++r) b[q][r] *= inv;
    var *= inv;
    double v[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}};
    for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
        bool rotated = jacobi_pair<0, 1>(b, v);
        rotated |= jacobi_pair<0, 2>(b, v);
        rotated |= jacobi_pair<1, 2>(b, v);
        if (!rotated) break;
    }
    double sig[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) sig[q] = sqrt(b[q][0] * b[q][0] + b[q][1] * b[q][1] + b[q][2] * b[q][2]);
    const int k = sig[2] <= sig[0] && sig[2] <= sig[1] ? 2 : sig[1] <= sig[0] ? 1 : 0;
    // selects, not b[(k + 1) % 3]: a run-time index would put the matrices in a local-memory stack frame
    double ui[3], uj[3], vi[3], vj[3], vk[3], bk[3];
    const double si = k == 0 ? sig[1] : k == 1 ? sig[2] : sig[0], sj = k == 0 ? sig[2] : k == 1 ? sig[0] : sig[1];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        ui[r] = (k == 0 ? b[1][r] : k == 1 ? b[2][r] : b[0][r]) / si;
        uj[r] = (k == 0 ? b[2][r] : k == 1 ? b[0][r] : b[1][r]) / sj;
        bk[r] = k == 0 ? b[0][r] : k == 1 ? b[1][r] : b[2][r];
        vi[r] = k == 0 ? v[1][r] : k == 1 ? v[2][r] : v[0][r];
        vj[r] = k == 0 ? v[2][r] : k == 1 ? v[0][r] : v[1][r];
        vk[r] = k == 0 ? v[0][r] : k == 1 ? v[1][r] : v[2][r];
    }
    const double w[3] = {ui[1] * uj[2] - ui[2] * uj[1], ui[2] * uj[0] - ui[0] * uj[2], ui[0] * uj[1] - ui[1] * uj[0]};
    const double c = with_scaling ? (si + sj + (bk[0] * w[0] + bk[1] * w[1] + bk[2] * w[2])) / var : 1.0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        double R[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) R[q] = ui[r] * vi[q] + uj[r] * vj[q] + w[r] * vk[q];
        T[4 * r] = c * R[0], T[4 * r + 1] = c * R[1], T[4 * r + 2] = c * R[2];
        T[4 * r + 3] = mt[r] - c * (R[0] * ms[0] + R[1] * ms[1] + R[2] * ms[2]);
    }
    return true;
}

__global__ void __launch_bounds__(kHypThreads) pc_ransac_hyp_kernel(const double* __restrict__ src, const double* __restrict__ tgt, int n,
                                                                   int n_hyp, int rn, double max_dist2, int with_scaling, uint64_t seed,
                                                                   int32_t* __restrict__ good_out, double* __restrict__ error2_out,
                                                                   double* __restrict__ trans_out, int32_t* __restrict__ samples) {
    __shared__ double ss[3][kAlignTile], st[3][kAlignTile];
    const int h = blockIdx.x * kHypThreads + threadIdx.x;
    double T[12];
    bool active = false;
    if (h < n_hyp) {
        active = ransac_umeyama(src, tgt, n, seed, h, rn, with_scaling, T);
        if (samples)
            for (int j = 0; j < rn; ++j) samples[(size_t)h * rn + j] = ransac_draw(seed, h, rn, j, n);
#pragma unroll
        for (int e = 0; e < 12; ++e) trans_out[(size_t)h * 12 + e] = active ? T[e] : __longlong_as_double(0x7ff8000000000000ll);
    }
    int good = 0;
    double error2 = 0.0;
    for (long long base = 0; base < n; base += kAlignTile) {
        const int cnt = n - base < kAlignTile ? (int)(n - base) : kAlignTile;
        __syncthreads();
        for (int t = threadIdx.x; t < 3 * cnt; t += kHypThreads) {
            const int p = t / 3, r = t - 3 * p;
            ss[r][p] = __ldg(src + 3 * base + t);
            st[r][p] = __ldg(tgt + 3 * base + t);
        }
        __syncthreads();
        if (!active) continue;
        for (int p = 0; p < cnt; ++p) {
            const double x = ss[0][p], y = ss[1][p], z = ss[2][p];
            double d[3];
#pragma unroll
            for (int r = 0; r < 3; ++r)
                d[r] = __dsub_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[4 * r], x), __dmul_rn(T[4 * r + 1], y)), __dmul_rn(T[4 * r + 2], z)),
                                           T[4 * r + 3]), st[r][p]);
            const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(d[0], d[0]), __dmul_rn(d[1], d[1])), __dmul_rn(d[2], d[2]));
            if (d2 < max_dist2) ++good, error2 = __dadd_rn(error2, d2);
        }
    }
    if (h < n_hyp) good_out[h] = good, error2_out[h] = error2;
}

struct Candidate {
    int good, h;
    double rmse;
};

// a beats b: more inliers, or as many with a smaller rmse, or both equal and an earlier hypothesis
__device__ __forceinline__ bool beats(const Candidate& a, const Candidate& b) {
    return a.good > b.good || (a.good == b.good && (a.rmse < b.rmse || (a.rmse == b.rmse && a.h < b.h)));
}

// record: [0] h (-1: no hypothesis has an inlier), [1] good, [2] error2, [3] rmse, [4..15] T (rows 0..2; the identity for h = -1),
// [16..16 + rn) the winner's draws
__global__ void __launch_bounds__(kSelectThreads) pc_ransac_select_kernel(const int32_t* __restrict__ good, const double* __restrict__ error2,
                                                                         const double* __restrict__ trans, int n_hyp, int n, int rn,
                                                                         uint64_t seed, double* __restrict__ record) {
    __shared__ int sg[kSelectThreads], sh[kSelectThreads];
    __shared__ double sr[kSelectThreads];
    const int t = threadIdx.x;
    Candidate best{0, -1, 0.0};
    for (int h = t; h < n_hyp; h += kSelectThreads) {
        const int g = good[h];
        if (g == 0) continue;
        const Candidate c{g, h, __dsqrt_rn(__ddiv_rn(error2[h], (double)g))};
        if (beats(c, best)) best = c;
    }
    sg[t] = best.good, sh[t] = best.h, sr[t] = best.rmse;
    __syncthreads();
    for (int w = kSelectThreads / 2; w > 0; w >>= 1) {
        if (t < w) {
            const Candidate o{sg[t + w], sh[t + w], sr[t + w]};
            if (beats(o, Candidate{sg[t], sh[t], sr[t]})) sg[t] = o.good, sh[t] = o.h, sr[t] = o.rmse;
        }
        __syncthreads();
    }
    const int h = sh[0];
    if (t == 0) record[0] = (double)h, record[1] = (double)sg[0], record[2] = h < 0 ? 0.0 : error2[h], record[3] = sr[0];
    if (t < 12) record[4 + t] = h < 0 ? (t % 5 == 0 ? 1.0 : 0.0) : trans[(size_t)h * 12 + t];
    if (t < rn) record[16 + t] = h < 0 ? -1.0 : (double)ransac_draw(seed, h, rn, t, n);
}

// ---- K10 normals: exact k-nearest neighbours on K8's grid and per-point normals (DESIGN §4 "K10 normals") --------------------------
// Each thread keeps its list ascending in (d^2, index) in dynamic shared memory laid out [slot][thread] (consecutive threads hit
// consecutive banks), k * kThreads floats of d^2 then as many ints of index.  kd, kj: the k-th entry once the list is full, and
// (lim, -1) before, so that "before (kd, kj)" is both the cap d^2 < max_dist^2 and the order test, and kd is the pruning bound.

constexpr int kKnnMax = MVSB200_PC_KNN_MAX;

// a candidate the order test admitted: insertion into the sorted list sd / si (this thread's slot 0) of cnt <= k entries
__device__ __forceinline__ void knn_insert(float d, int j, float* sd, int* si, int k, int& cnt, float& kd, int& kj) {
    int p = cnt < k ? cnt : k - 1;
    for (; p > 0; --p) {
        const float pd = sd[(p - 1) * kThreads];
        const int pj = si[(p - 1) * kThreads];
        if (pd < d || (pd == d && pj < j)) break;
        sd[p * kThreads] = pd, si[p * kThreads] = pj;
    }
    sd[p * kThreads] = d, si[p * kThreads] = j;
    if (cnt < k) ++cnt;
    if (cnt == k) kd = sd[(k - 1) * kThreads], kj = si[(k - 1) * kThreads];
}

// scan_points for the list: the candidates the order test admits are inserted
__device__ __forceinline__ void knn_scan(const float4* __restrict__ pts, int b, int e, float qx, float qy, float qz, float* sd, int* si,
                                         int k, int& cnt, float& kd, int& kj) {
    for (int p = b; p < e; ++p) {
        const float4 t = __ldg(pts + p);
        const float d = sq(t.x - qx) + sq(t.y - qy) + sq(t.z - qz);
        const int j = __float_as_int(t.w);
        if (d < kd || (d == kd && j < kj)) knn_insert(d, j, sd, si, k, cnt, kd, kj);
    }
}

// NORMALS = false: dist / index [n, k].  NORMALS = true: query is also the grid's cloud (index j -> query[3 j ..]); normals [n, 3]
// from the list, which is never written out.  view_mode 0: none, 1: view[0..2], 2: view[3 i ..].
template <bool NORMALS>
__global__ void __launch_bounds__(kThreads, 2) pc_knn_kernel(const float* __restrict__ query, int n, const float4* __restrict__ pts,
                                                          const int2* __restrict__ cells, const int2* __restrict__ blocks, Grid g,
                                                          float slack, float max_dist, int k, float* __restrict__ dist,
                                                          int32_t* __restrict__ index, const double* __restrict__ view, int view_mode,
                                                          float* __restrict__ normals) {
    extern __shared__ float knn_smem[];
    float* sd = knn_smem + threadIdx.x;
    int* si = reinterpret_cast<int*>(knn_smem + k * kThreads) + threadIdx.x;
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const float qx = query[3 * (size_t)i], qy = query[3 * (size_t)i + 1], qz = query[3 * (size_t)i + 2];
    const int nx = 8 * g.nbx, ny = 8 * g.nby, nz = 8 * g.nbz;
    const float lim = max_dist * max_dist;
    // the list's count and k-th entry: as one object the kernel takes 61 registers, as three locals 62
    struct { int cnt; float kd; int kj; } top{0, lim, -1};
    if (box_gap2(qx, qy, qz, g, nx, ny, nz) < (double)max_dist * max_dist) {
        const float sl = slack + 2.4e-7f * (fabsf(qx) + fabsf(qy) + fabsf(qz));
        const int cx = cell_of(qx, g.ox, g.inv, nx), cy = cell_of(qy, g.oy, g.inv, ny), cz = cell_of(qz, g.oz, g.inv, nz);
        grid_search<true>(qx, qy, qz, cx, cy, cz, g, sl, cells, blocks, [&] { return top.kd; },
                          [&](int b, int e) { knn_scan(pts, b, e, qx, qy, qz, sd, si, k, top.cnt, top.kd, top.kj); });
    }
    // the cap on the distance itself: the list is cut at the first entry whose root is not below max_dist
    int c = 0;
    for (; c < top.cnt; ++c)
        if (!(root_below(sd[c * kThreads], lim) < max_dist)) break;
    if constexpr (!NORMALS) {
        for (int s = 0; s < k; ++s) {
            dist[(size_t)i * k + s] = s < c ? root_below(sd[s * kThreads], lim) : kInf;
            index[(size_t)i * k + s] = s < c ? si[s * kThreads] : -1;
        }
    } else {
        double nrm[3] = {0.0, 0.0, 0.0};
        if (c >= 3) {
            double mx = 0.0, my = 0.0, mz = 0.0;
            for (int s = 0; s < c; ++s) {
                const size_t j = (size_t)si[s * kThreads];
                mx += __ldg(query + 3 * j), my += __ldg(query + 3 * j + 1), mz += __ldg(query + 3 * j + 2);
            }
            mx /= c, my /= c, mz /= c;
            double b[3][3] = {};                        // b[q][r] = C[r][q]: column q (C is symmetric)
            for (int s = 0; s < c; ++s) {
                const size_t j = (size_t)si[s * kThreads];
                const double dx = __ldg(query + 3 * j) - mx, dy = __ldg(query + 3 * j + 1) - my, dz = __ldg(query + 3 * j + 2) - mz;
                b[0][0] += dx * dx, b[0][1] += dx * dy, b[0][2] += dx * dz;
                b[1][1] += dy * dy, b[1][2] += dy * dz, b[2][2] += dz * dz;
            }
            b[0][0] /= c, b[0][1] /= c, b[0][2] /= c, b[1][1] /= c, b[1][2] /= c, b[2][2] /= c;
            b[1][0] = b[0][1], b[2][0] = b[0][2], b[2][1] = b[1][2];
            if (b[0][0] + b[1][1] + b[2][2] > 0.0) {
                // one-sided Jacobi on C's columns: B = C V with orthogonal columns b_q = lambda_q v_q, so for C positive semi-definite
                // the column of V under the smallest |b_q| is the eigenvector of the smallest eigenvalue
                double v[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}};
                for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
                    bool rotated = jacobi_pair<0, 1>(b, v);
                    rotated |= jacobi_pair<0, 2>(b, v);
                    rotated |= jacobi_pair<1, 2>(b, v);
                    if (!rotated) break;
                }
                double s2[3];
#pragma unroll
                for (int q = 0; q < 3; ++q) s2[q] = b[q][0] * b[q][0] + b[q][1] * b[q][1] + b[q][2] * b[q][2];
                const int q = s2[2] <= s2[0] && s2[2] <= s2[1] ? 2 : s2[1] <= s2[0] ? 1 : 0;
                // selects, not v[q]: a run-time index would put v in a local-memory stack frame
#pragma unroll
                for (int r = 0; r < 3; ++r) nrm[r] = q == 0 ? v[0][r] : q == 1 ? v[1][r] : v[2][r];
                const double ax = fabs(nrm[0]), ay = fabs(nrm[1]), az = fabs(nrm[2]);
                const double big = ax >= ay && ax >= az ? nrm[0] : ay >= az ? nrm[1] : nrm[2];
                double sgn = big < 0.0 ? -1.0 : 1.0;
                if (view_mode) {
                    const size_t o = view_mode == 2 ? 3 * (size_t)i : 0;
                    const double dot = sgn * (nrm[0] * (__ldg(view + o) - qx) + nrm[1] * (__ldg(view + o + 1) - qy) +
                                              nrm[2] * (__ldg(view + o + 2) - qz));
                    if (dot < 0.0) sgn = -sgn;
                }
#pragma unroll
                for (int r = 0; r < 3; ++r) nrm[r] *= sgn;
            }
        }
#pragma unroll
        for (int r = 0; r < 3; ++r) normals[3 * (size_t)i + r] = (float)nrm[r];
    }
}

int blocks_for(int n) { return (n + kThreads - 1) / kThreads; }

bool grid_ok(float cell, int nbx, int nby, int nbz) {
    return cell > 0.f && isfinite(cell) && nbx >= 1 && nby >= 1 && nbz >= 1 &&
           (long long)nbx * nby * nbz * 512 <= (long long)MVSB200_PC_MAX_CELLS;
}

// the checks of a search on a built grid (float4 points, int2 cells and blocks; blocks may be null) -> g
int search_grid(const char* what, const float* pts, const int32_t* cells, const int32_t* blocks, float ox, float oy, float oz,
                float cell, int nbx, int nby, int nbz, Grid& g) {
    MVS_REQUIRE(aligned16(pts) && ((uintptr_t)cells & 7) == 0 && ((uintptr_t)blocks & 7) == 0, "%s: misaligned buffer", what);
    MVS_REQUIRE(grid_ok(cell, nbx, nby, nbz), "%s: cell > 0 and at most %d cells", what, MVSB200_PC_MAX_CELLS);
    g = Grid{ox, oy, oz, cell, nbx, nby, nbz, 1.0 / (double)cell};
    return MVSB200_OK;
}

template <bool IDX>
int nearest_launch(const char* what, const float* query, int n, const float* pts, const int32_t* cells, const int32_t* blocks, float ox,
                   float oy, float oz, float cell, int nbx, int nby, int nbz, float slack, float max_dist, float* dist, int32_t* index,
                   void* stream) {
    MVS_REQUIRE(n >= 0, "%s: 0 <= n < 2^31 queries", what);
    Grid g;
    const int rc = search_grid(what, pts, cells, blocks, ox, oy, oz, cell, nbx, nby, nbz, g);
    if (rc != MVSB200_OK) return rc;
    MVS_REQUIRE(max_dist > 0.f && isfinite(max_dist) && slack >= 0.f, "%s: max_dist > 0 (finite), slack >= 0", what);
    if (n == 0) return MVSB200_OK;
    pc_nearest_kernel<IDX><<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(query, n, (const float4*)pts, (const int2*)cells,
                                                                                 (const int2*)blocks, g, slack, max_dist, dist, index);
    MVS_CHECK_LAUNCH(what);
    return MVSB200_OK;
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
    return nearest_launch<false>("pc_nearest", query, n, pts, cells, blocks, ox, oy, oz, cell, nbx, nby, nbz, slack, max_dist, dist,
                                 nullptr, stream);
}

extern "C" int mvsb200_pc_nearest_index(const float* query, int n, const float* pts, const int32_t* cells, const int32_t* blocks,
                                        float ox, float oy, float oz, float cell, int nbx, int nby, int nbz, float slack, float max_dist,
                                        float* dist, int32_t* index, void* stream) {
    MVS_REQUIRE(query && pts && cells && blocks && dist && index, "pc_nearest_index: null pointer");
    return nearest_launch<true>("pc_nearest_index", query, n, pts, cells, blocks, ox, oy, oz, cell, nbx, nby, nbz, slack, max_dist, dist,
                                index, stream);
}

extern "C" int mvsb200_pc_thin_neighbours(const float* pts, const int32_t* cells, const int32_t* rank_sorted, int n, float ox, float oy,
                                          float oz, float cell, int nbx, int nby, int nbz, double dst, const int64_t* offsets,
                                          int32_t* counts, int32_t* list, void* stream) {
    MVS_REQUIRE(pts && cells && rank_sorted, "pc_thin_neighbours: null pointer");
    MVS_REQUIRE(offsets ? list != nullptr : counts != nullptr, "pc_thin_neighbours: counts, or offsets and list");
    MVS_REQUIRE(n >= 1, "pc_thin_neighbours: 1 <= n < 2^31 points");
    Grid g;
    const int rc = search_grid("pc_thin_neighbours", pts, cells, nullptr, ox, oy, oz, cell, nbx, nby, nbz, g);
    if (rc != MVSB200_OK) return rc;
    MVS_REQUIRE(dst > 0.0 && (double)cell >= dst, "pc_thin_neighbours: 0 < dst <= cell");
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

extern "C" int mvsb200_pc_transform_crop(const float* xyz, int n, const double* affine12_host, const double* polygon, int k, int axis,
                                         double axis_min, double axis_max, double* out, uint8_t* keep, void* stream) {
    MVS_REQUIRE(xyz && polygon && out && keep, "pc_transform_crop: null pointer");
    MVS_REQUIRE(n >= 1, "pc_transform_crop: 1 <= n < 2^31 points");
    MVS_REQUIRE(k >= 3 && k <= kMaxPolygon, "pc_transform_crop: a polygon of 3 to %d vertices, got %d", kMaxPolygon, k);
    MVS_REQUIRE(axis >= 0 && axis <= 2, "pc_transform_crop: orthogonal axis 0, 1 or 2, got %d", axis);
    MVS_REQUIRE(isfinite(axis_min) && isfinite(axis_max), "pc_transform_crop: finite axis bounds");
    Affine A{};
    if (affine12_host) {
        for (int t = 0; t < 12; ++t) {
            MVS_REQUIRE(isfinite(affine12_host[t]), "pc_transform_crop: the transform must be finite");
            A.a[t] = affine12_host[t];
        }
    }
    // (u, v, w) of Open3D's CropInPolygon: x -> (1, 2, 0), y -> (0, 2, 1), z -> (0, 1, 2)
    const int u = axis == 0 ? 1 : 0, v = axis == 2 ? 1 : 2;
    pc_transform_crop_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(xyz, n, A, affine12_host != nullptr, polygon, k, u, v,
                                                                                   axis, axis_min, axis_max, out, keep);
    MVS_CHECK_LAUNCH("pc_transform_crop");
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_voxel_keys(const double* xyz, int n, double ox, double oy, double oz, double voxel, int64_t nx, int64_t ny,
                                     int64_t nz, int64_t* keys, void* stream) {
    MVS_REQUIRE(xyz && keys, "pc_voxel_keys: null pointer");
    MVS_REQUIRE(n >= 1, "pc_voxel_keys: 1 <= n < 2^31 points");
    MVS_REQUIRE(voxel > 0.0 && isfinite(voxel) && isfinite(ox) && isfinite(oy) && isfinite(oz), "pc_voxel_keys: voxel > 0, finite origin");
    MVS_REQUIRE(nx >= 1 && ny >= 1 && nz >= 1 && nx < (int64_t(1) << 62) / ny && nx * ny < (int64_t(1) << 62) / nz,
                "pc_voxel_keys: 1 <= voxels per axis and nx ny nz < 2^62");
    pc_voxel_keys_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(xyz, n, ox, oy, oz, voxel, nx, ny, keys);
    MVS_CHECK_LAUNCH("pc_voxel_keys");
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_voxel_mean(const double* xyz, const int64_t* perm, const int64_t* offsets, int n_voxels, double* mean,
                                     float* mean_f32, void* stream) {
    MVS_REQUIRE(xyz && perm && offsets && mean && mean_f32, "pc_voxel_mean: null pointer");
    MVS_REQUIRE(n_voxels >= 1, "pc_voxel_mean: 1 <= n_voxels < 2^31");
    pc_voxel_mean_kernel<<<blocks_for(n_voxels), kThreads, 0, (cudaStream_t)stream>>>(xyz, perm, offsets, n_voxels, mean, mean_f32);
    MVS_CHECK_LAUNCH("pc_voxel_mean");
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_icp_sums(const double* src, const int32_t* index, int n, const double* tgt, double* partial, uint32_t* ticket,
                                   double* sums, void* stream) {
    MVS_REQUIRE(src && index && tgt && partial && ticket && sums, "pc_icp_sums: null pointer");
    MVS_REQUIRE(n >= 1, "pc_icp_sums: 1 <= n < 2^31 source points");
    const int nb = blocks_for(n) < kSumBlocks ? blocks_for(n) : kSumBlocks;
    pc_icp_sums_a_kernel<<<nb, kThreads, 0, (cudaStream_t)stream>>>(src, index, n, tgt, partial, sums, ticket);
    MVS_CHECK_LAUNCH("pc_icp_sums_a");
    pc_icp_sums_b_kernel<<<nb, kThreads, 0, (cudaStream_t)stream>>>(src, index, n, tgt, partial, sums, ticket + 1);
    MVS_CHECK_LAUNCH("pc_icp_sums_b");
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_transform64(double* xyz, int n, const double* affine12_host, float* xyz_f32, void* stream) {
    MVS_REQUIRE(xyz && affine12_host && xyz_f32, "pc_transform64: null pointer");
    MVS_REQUIRE(n >= 1, "pc_transform64: 1 <= n < 2^31 points");
    Affine A{};
    for (int t = 0; t < 12; ++t) {
        MVS_REQUIRE(isfinite(affine12_host[t]), "pc_transform64: the transform must be finite");
        A.a[t] = affine12_host[t];
    }
    pc_transform64_kernel<<<blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(xyz, n, A, xyz_f32);
    MVS_CHECK_LAUNCH("pc_transform64");
    return MVSB200_OK;
}

extern "C" int mvsb200_pc_ransac_align(const double* src, const double* tgt, int n, int n_hyp, int ransac_n, double max_dist2,
                                       int with_scaling, uint64_t seed, int32_t* good, double* error2, double* trans, int32_t* samples,
                                       double* record, void* stream) {
    MVS_REQUIRE(src && tgt && good && error2 && trans && record, "pc_ransac_align: null pointer");
    MVS_REQUIRE(n >= 1, "pc_ransac_align: 1 <= n < 2^31 correspondences");
    MVS_REQUIRE(n_hyp >= 1, "pc_ransac_align: 1 <= n_hyp < 2^31 hypotheses");
    MVS_REQUIRE(ransac_n >= 3 && ransac_n <= kMaxSample, "pc_ransac_align: 3 <= ransac_n <= %d, got %d", kMaxSample, ransac_n);
    MVS_REQUIRE(max_dist2 > 0.0 && isfinite(max_dist2), "pc_ransac_align: max_dist2 > 0 (finite)");
    pc_ransac_hyp_kernel<<<(n_hyp + kHypThreads - 1) / kHypThreads, kHypThreads, 0, (cudaStream_t)stream>>>(
        src, tgt, n, n_hyp, ransac_n, max_dist2, with_scaling != 0, seed, good, error2, trans, samples);
    MVS_CHECK_LAUNCH("pc_ransac_hyp");
    pc_ransac_select_kernel<<<1, kSelectThreads, 0, (cudaStream_t)stream>>>(good, error2, trans, n_hyp, n, ransac_n, seed, record);
    MVS_CHECK_LAUNCH("pc_ransac_select");
    return MVSB200_OK;
}

namespace {

template <bool NORMALS>
int knn_launch(const char* what, const float* query, int n, const float* pts, const int32_t* cells, const int32_t* blocks, float ox,
               float oy, float oz, float cell, int nbx, int nby, int nbz, float slack, float max_dist, int k, float* dist,
               int32_t* index, const double* view, int view_mode, float* normals, void* stream) {
    MVS_REQUIRE(n >= 0, "%s: 0 <= n < 2^31 queries", what);
    Grid g;
    const int rc = search_grid(what, pts, cells, blocks, ox, oy, oz, cell, nbx, nby, nbz, g);
    if (rc != MVSB200_OK) return rc;
    MVS_REQUIRE(max_dist > 0.f && slack >= 0.f, "%s: max_dist > 0 (+inf allowed), slack >= 0", what);
    MVS_REQUIRE(k >= 1 && k <= kKnnMax, "%s: 1 <= k <= %d, got %d", what, kKnnMax, k);
    if (n == 0) return MVSB200_OK;
    const int smem = k * kThreads * (int)(sizeof(float) + sizeof(int));
    MVS_CUDA(cudaFuncSetAttribute(pc_knn_kernel<NORMALS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    pc_knn_kernel<NORMALS><<<blocks_for(n), kThreads, smem, (cudaStream_t)stream>>>(
        query, n, (const float4*)pts, (const int2*)cells, (const int2*)blocks, g, slack, max_dist, k, dist, index, view, view_mode, normals);
    MVS_CHECK_LAUNCH(what);
    return MVSB200_OK;
}

}  // namespace

extern "C" int mvsb200_pc_knn(const float* query, int n, const float* pts, const int32_t* cells, const int32_t* blocks, float ox, float oy,
                              float oz, float cell, int nbx, int nby, int nbz, float slack, float max_dist, int k, float* dist,
                              int32_t* index, void* stream) {
    MVS_REQUIRE(query && pts && cells && blocks && dist && index, "pc_knn: null pointer");
    return knn_launch<false>("pc_knn", query, n, pts, cells, blocks, ox, oy, oz, cell, nbx, nby, nbz, slack, max_dist, k, dist, index,
                             nullptr, 0, nullptr, stream);
}

extern "C" int mvsb200_pc_normals(const float* xyz, int n, const float* pts, const int32_t* cells, const int32_t* blocks, float ox,
                                  float oy, float oz, float cell, int nbx, int nby, int nbz, float slack, float max_dist, int k,
                                  const double* viewpoints, int view_mode, float* normals, void* stream) {
    MVS_REQUIRE(xyz && pts && cells && blocks && normals, "pc_normals: null pointer");
    MVS_REQUIRE(view_mode >= 0 && view_mode <= 2, "pc_normals: view_mode 0, 1 or 2, got %d", view_mode);
    MVS_REQUIRE(view_mode == 0 || viewpoints, "pc_normals: view_mode %d needs viewpoints", view_mode);
    return knn_launch<true>("pc_normals", xyz, n, pts, cells, blocks, ox, oy, oz, cell, nbx, nby, nbz, slack, max_dist, k, nullptr,
                            nullptr, viewpoints, view_mode, normals, stream);
}
