// Isosurface of a scalar grid by marching tetrahedra on the Kuhn (Freudenthal) split, for mesh export of a trained
// density field (NeRF.extract_mesh).  Rules (restated by the NumPy reference tests/mesh_oracle.py, which the GPU
// tests compare against index for index):
//  * field[(i*ny + j)*nz + k], x slowest; a grid point is INSIDE when f > iso (strict).
//  * every cell (i < nx-1, j < ny-1, k < nz-1) splits into 6 tets 0 -> e_a -> e_a+e_b -> 111, one per axis permutation
//    (a,b,c) in the order kPerm below.  The split is the same in every cell, so neighbouring tets share faces and the
//    surface is watertight without a case table.
//  * every tet edge runs from a grid point p to p + delta, delta one of the 7 offsets of kDelta; p owns the edge, and
//    its vertex when exactly one endpoint is inside: t = (iso - f_p) / (f_q - f_p), v = origin + spacing * (p + t delta).
//    Normal: the central-difference gradient (one-sided on the grid faces) at both endpoints interpolated with the same
//    t, normalised and negated (towards decreasing f); a zero gradient gives a zero normal.
//  * a tet with 1 or 3 corners inside gives one triangle, with 2 inside (a, b) and 2 outside (c, d) the quad
//    ac, ad, bd, bc split along ac-bd.  Orientation from the EDGE MIDPOINTS (half-integer, exact in integers here): the
//    triangle's normal points from the centroid of the inside corners to the outside ones.
//  * output order: vertices by (point, delta index), triangles by (cell, tet, triangle); no atomics, so two runs give
//    the same bytes.
//
// Two passes.  Count: one block per tile of kTile consecutive points classifies them, stores per point the 7-bit mask
// of its crossing edges and the in-tile exclusive prefix of the vertex and triangle counts (uint16: at most 7 / 12 per
// point), then one block scans the per-tile totals into int64 tile offsets.  Emit: one thread per point recomputes
// its classification from the field and writes its vertices and its cell's triangles at offset(tile) + prefix; the
// vertex index of a neighbour's edge is offset(tile of q) + prefix(q) + popcount of q's lower crossing bits.
// Workspace: 5 bytes per grid point + 24 per tile; the field is read once per pass (plus the gradient stencil of the
// crossing edges).
#include "common.cuh"

namespace knerf {
namespace {

constexpr int kThreads = 256;
constexpr int kItems = 8;
constexpr int kTile = kThreads * kItems;   // points per tile: counts <= 12 * 2048 < 2^16 fit the uint16 prefixes
constexpr int kScanThreads = 1024;

// (dx,dy,dz) of the 7 edge offsets, in vertex order 100, 010, 001, 110, 101, 011, 111
__constant__ int8_t kDelta[7][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}, {1, 1, 0}, {1, 0, 1}, {0, 1, 1}, {1, 1, 1}};
// delta index of the offset with bits 4*dx + 2*dy + dz
__constant__ int8_t kDeltaIndex[8] = {-1, 2, 1, 5, 0, 4, 3, 6};
// the 6 axis permutations (a, b, c): tet corners 0, e_a, e_a + e_b, 111
__constant__ int8_t kPerm[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};

struct Grid {
  int nx, ny, nz;
  int64_t n;   // nx * ny * nz
};

struct Workspace {
  uint8_t* mask;       // [n] crossing-edge bits of every point
  uint16_t* vloc;      // [n] in-tile exclusive prefix of the vertex counts
  uint16_t* tloc;      // [n] in-tile exclusive prefix of the triangle counts
  int32_t* tile_sum;   // [tiles][2] per-tile vertex / triangle totals
  int64_t* tile_off;   // [tiles][2] exclusive prefix of tile_sum
};

__device__ __forceinline__ void corner_of_tet(int tet, int v, int (&c)[3]) {
  c[0] = c[1] = c[2] = (v == 3) ? 1 : 0;
  if (v == 1 || v == 2) c[kPerm[tet][0]] = 1;
  if (v == 2) c[kPerm[tet][1]] = 1;
}

// the 8 corner values of the cell at (i,j,k) as inside bits (bit 4*dx + 2*dy + dz), corners past the grid outside
__device__ __forceinline__ unsigned corner_bits(const float* __restrict__ f, const Grid& g, int i, int j, int k,
                                                int64_t p, float iso) {
  unsigned bits = 0;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int dx = c >> 2, dy = (c >> 1) & 1, dz = c & 1;
    if (i + dx < g.nx && j + dy < g.ny && k + dz < g.nz &&
        __ldg(f + p + ((int64_t)dx * g.ny + dy) * g.nz + dz) > iso)
      bits |= 1u << c;
  }
  return bits;
}

__device__ __forceinline__ unsigned crossing_mask(unsigned bits, const Grid& g, int i, int j, int k) {
  unsigned m = 0;
  const bool in0 = bits & 1u;
#pragma unroll
  for (int d = 0; d < 7; ++d) {
    const int dx = kDelta[d][0], dy = kDelta[d][1], dz = kDelta[d][2];
    if (i + dx < g.nx && j + dy < g.ny && k + dz < g.nz && (((bits >> (4 * dx + 2 * dy + dz)) & 1u) != in0))
      m |= 1u << d;
  }
  return m;
}

// inside bits of the 4 corners of tet `tet` from the cell's corner bits
__device__ __forceinline__ unsigned tet_bits(unsigned cell_bits, int tet) {
  unsigned b = 0;
#pragma unroll
  for (int v = 0; v < 4; ++v) {
    int c[3];
    corner_of_tet(tet, v, c);
    b |= ((cell_bits >> (4 * c[0] + 2 * c[1] + c[2])) & 1u) << v;
  }
  return b;
}

__device__ __forceinline__ int tris_of(unsigned tb) {
  const int n = __popc(tb);
  return (n == 1 || n == 3) ? 1 : (n == 2 ? 2 : 0);
}

__device__ __forceinline__ bool cell_valid(const Grid& g, int i, int j, int k) {
  return i < g.nx - 1 && j < g.ny - 1 && k < g.nz - 1;
}

__device__ __forceinline__ void coords(const Grid& g, int64_t p, int& i, int& j, int& k) {
  k = (int)(p % g.nz);
  const int64_t r = p / g.nz;
  j = (int)(r % g.ny);
  i = (int)(r / g.ny);
}

// exclusive block scan of one int per thread (kThreads threads); returns the block total in *total
__device__ __forceinline__ int block_exclusive_scan(int v, int* total) {
  __shared__ int warp_tot[kThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int n = __shfl_up_sync(kFullMask, inc, o);
    if (lane >= o) inc += n;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  int before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    before += (w < warp) ? warp_tot[w] : 0;
    all += warp_tot[w];
  }
  *total = all;
  return before + inc - v;
}

__global__ void __launch_bounds__(kThreads) iso_count_kernel(const float* __restrict__ f, Grid g, float iso,
                                                             Workspace ws) {
  const int64_t base = (int64_t)blockIdx.x * kTile + (int64_t)threadIdx.x * kItems;
  uint8_t m[kItems];
  uint8_t nt[kItems];
  int sv = 0, st = 0;
#pragma unroll
  for (int u = 0; u < kItems; ++u) {
    const int64_t p = base + u;
    m[u] = 0;
    nt[u] = 0;
    if (p < g.n) {
      int i, j, k;
      coords(g, p, i, j, k);
      const unsigned bits = corner_bits(f, g, i, j, k, p, iso);
      m[u] = (uint8_t)crossing_mask(bits, g, i, j, k);
      if (cell_valid(g, i, j, k) && bits != 0 && bits != 0xffu) {
        int n = 0;
#pragma unroll
        for (int tet = 0; tet < 6; ++tet) n += tris_of(tet_bits(bits, tet));
        nt[u] = (uint8_t)n;
      }
    }
    sv += __popc(m[u]);
    st += nt[u];
  }
  // vertex counts in the low 16 bits, triangle counts in the high ones: each tile total is < 2^15
  int total;
  const int before = block_exclusive_scan(sv | (st << 16), &total);
  int v = before & 0xffff, t = before >> 16;
#pragma unroll
  for (int u = 0; u < kItems; ++u) {
    const int64_t p = base + u;
    if (p < g.n) {
      ws.mask[p] = m[u];
      ws.vloc[p] = (uint16_t)v;
      ws.tloc[p] = (uint16_t)t;
    }
    v += __popc(m[u]);
    t += nt[u];
  }
  if (threadIdx.x == 0) {
    ws.tile_sum[2 * blockIdx.x] = total & 0xffff;
    ws.tile_sum[2 * blockIdx.x + 1] = total >> 16;
  }
}

// one block: exclusive int64 scan of the per-tile (V, T) totals, in rounds of kScanThreads * kItems tiles
__global__ void __launch_bounds__(kScanThreads) iso_scan_kernel(Workspace ws, int64_t tiles, int64_t* counts) {
  __shared__ long long warp_tot[2][kScanThreads / 32];
  __shared__ long long carry[2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry[0] = carry[1] = 0;
  for (int64_t r0 = 0; r0 < tiles; r0 += (int64_t)kScanThreads * kItems) {
    const int64_t b = r0 + (int64_t)threadIdx.x * kItems;
    long long s[2] = {0, 0};
#pragma unroll
    for (int u = 0; u < kItems; ++u)
      if (b + u < tiles) {
        s[0] += ws.tile_sum[2 * (b + u)];
        s[1] += ws.tile_sum[2 * (b + u) + 1];
      }
    long long inc[2] = {s[0], s[1]};
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long n0 = __shfl_up_sync(kFullMask, inc[0], o), n1 = __shfl_up_sync(kFullMask, inc[1], o);
      if (lane >= o) { inc[0] += n0; inc[1] += n1; }
    }
    __syncthreads();   // carry and warp_tot of the previous round are read
    if (lane == 31) { warp_tot[0][warp] = inc[0]; warp_tot[1][warp] = inc[1]; }
    __syncthreads();
    long long run[2] = {carry[0], carry[1]}, all[2] = {0, 0};
    for (int w = 0; w < kScanThreads / 32; ++w)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (w < warp) run[h] += warp_tot[h][w];
        all[h] += warp_tot[h][w];
      }
#pragma unroll
    for (int h = 0; h < 2; ++h) run[h] += inc[h] - s[h];
#pragma unroll
    for (int u = 0; u < kItems; ++u)
      if (b + u < tiles) {
        ws.tile_off[2 * (b + u)] = run[0];
        ws.tile_off[2 * (b + u) + 1] = run[1];
        run[0] += ws.tile_sum[2 * (b + u)];
        run[1] += ws.tile_sum[2 * (b + u) + 1];
      }
    __syncthreads();
    if (threadIdx.x == 0) { carry[0] += all[0]; carry[1] += all[1]; }
  }
  __syncthreads();
  if (threadIdx.x == 0) { counts[0] = carry[0]; counts[1] = carry[1]; }
}

// central difference along `axis` at grid coordinate x of n (one-sided on the faces), in field units per world unit
__device__ __forceinline__ float grad1(const float* __restrict__ f, int64_t p, int64_t stride, int x, int n, float h) {
  if (x == 0) return __fdiv_rn(__fsub_rn(__ldg(f + p + stride), __ldg(f + p)), h);
  if (x == n - 1) return __fdiv_rn(__fsub_rn(__ldg(f + p), __ldg(f + p - stride)), h);
  return __fdiv_rn(__fsub_rn(__ldg(f + p + stride), __ldg(f + p - stride)), __fmul_rn(2.f, h));
}

struct Frame {
  float origin[3], spacing[3];
};

__device__ __forceinline__ int64_t vertex_index(const Workspace& ws, int64_t q, int d) {
  return ws.tile_off[2 * (q / kTile)] + ws.vloc[q] + __popc(ws.mask[q] & ((1u << d) - 1u));
}

__global__ void __launch_bounds__(kThreads) iso_emit_kernel(const float* __restrict__ f, Grid g, float iso, Frame fr,
                                                            Workspace ws, float* __restrict__ vertices,
                                                            float* __restrict__ normals, int32_t* __restrict__ tris,
                                                            int64_t max_v, int64_t max_t) {
  const int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (p >= g.n) return;
  int i, j, k;
  coords(g, p, i, j, k);
  const int64_t sx = (int64_t)g.ny * g.nz, sy = g.nz;
  const unsigned mask = ws.mask[p];
  if (mask) {
    int64_t v = ws.tile_off[2 * (p / kTile)] + ws.vloc[p];
    const float fp = __ldg(f + p);
    float gp[3];
    if (normals) {
      gp[0] = grad1(f, p, sx, i, g.nx, fr.spacing[0]);
      gp[1] = grad1(f, p, sy, j, g.ny, fr.spacing[1]);
      gp[2] = grad1(f, p, 1, k, g.nz, fr.spacing[2]);
    }
    for (int d = 0; d < 7; ++d) {
      if (!((mask >> d) & 1u)) continue;
      const int dx = kDelta[d][0], dy = kDelta[d][1], dz = kDelta[d][2];
      const int64_t q = p + dx * sx + dy * sy + dz;
      const float t = __fdiv_rn(__fsub_rn(iso, fp), __fsub_rn(__ldg(f + q), fp));
      if (v < max_v) {
        const int pc[3] = {i, j, k}, dc[3] = {dx, dy, dz};
#pragma unroll
        for (int c = 0; c < 3; ++c)
          vertices[3 * v + c] = __fadd_rn(fr.origin[c], __fmul_rn(fr.spacing[c], __fadd_rn((float)pc[c],
                                                                                            __fmul_rn(t, (float)dc[c]))));
        if (normals) {
          const float gq[3] = {grad1(f, q, sx, i + dx, g.nx, fr.spacing[0]), grad1(f, q, sy, j + dy, g.ny, fr.spacing[1]),
                               grad1(f, q, 1, k + dz, g.nz, fr.spacing[2])};
          float n[3];
#pragma unroll
          for (int c = 0; c < 3; ++c) n[c] = __fadd_rn(gp[c], __fmul_rn(t, __fsub_rn(gq[c], gp[c])));
          const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(n[0], n[0]), __fmul_rn(n[1], n[1])),
                                                 __fmul_rn(n[2], n[2])));
#pragma unroll
          for (int c = 0; c < 3; ++c) normals[3 * v + c] = len > 0.f ? -__fdiv_rn(n[c], len) : 0.f;
        }
      }
      ++v;
    }
  }
  if (!cell_valid(g, i, j, k)) return;
  const unsigned bits = corner_bits(f, g, i, j, k, p, iso);
  if (bits == 0 || bits == 0xffu) return;
  int64_t tri = ws.tile_off[2 * (p / kTile) + 1] + ws.tloc[p];
  for (int tet = 0; tet < 6; ++tet) {
    const unsigned tb = tet_bits(bits, tet);
    const int nin = __popc(tb);
    if (nin == 0 || nin == 4) continue;
    int cs[4][3];
#pragma unroll
    for (int v = 0; v < 4; ++v) corner_of_tet(tet, v, cs[v]);
    int in[3], out[3], ni = 0, no = 0;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      if ((tb >> v) & 1u) in[ni++] = v;
      else out[no++] = v;
    }
    // the triangles as pairs of tet corners (edge list), before orientation
    int e[2][3][2], ntri;
    if (nin == 1) {
      ntri = 1;
      for (int m = 0; m < 3; ++m) { e[0][m][0] = in[0]; e[0][m][1] = out[m]; }
    } else if (nin == 3) {
      ntri = 1;
      for (int m = 0; m < 3; ++m) { e[0][m][0] = in[m]; e[0][m][1] = out[0]; }
    } else {   // a, b inside, c, d outside: (ac, ad, bd), (ac, bd, bc)
      ntri = 2;
      const int a = in[0], b = in[1], c = out[0], dd = out[1];
      e[0][0][0] = a; e[0][0][1] = c;  e[0][1][0] = a; e[0][1][1] = dd; e[0][2][0] = b; e[0][2][1] = dd;
      e[1][0][0] = a; e[1][0][1] = c;  e[1][1][0] = b; e[1][1][1] = dd; e[1][2][0] = b; e[1][2][1] = c;
    }
    // inside -> outside direction, scaled by ni * no > 0: no * sum(in) vs ni * sum(out)
    int dir[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      int si = 0, so = 0;
      for (int v = 0; v < 4; ++v) {
        if ((tb >> v) & 1u) si += cs[v][c];
        else so += cs[v][c];
      }
      dir[c] = ni * so - no * si;
    }
    for (int s = 0; s < ntri; ++s, ++tri) {
      int mid[3][3];   // doubled edge midpoints
      int64_t idx[3];
      for (int m = 0; m < 3; ++m) {
        int lo = e[s][m][0], hi = e[s][m][1];
        if (lo > hi) { const int x = lo; lo = hi; hi = x; }   // corners along the chain: lower index = base point
        const int* cl = cs[lo];
        const int* ch = cs[hi];
        for (int c = 0; c < 3; ++c) mid[m][c] = cl[c] + ch[c];
        const int64_t q = p + cl[0] * sx + cl[1] * sy + cl[2];
        idx[m] = vertex_index(ws, q, kDeltaIndex[4 * (ch[0] - cl[0]) + 2 * (ch[1] - cl[1]) + (ch[2] - cl[2])]);
      }
      const int u0 = mid[1][0] - mid[0][0], u1 = mid[1][1] - mid[0][1], u2 = mid[1][2] - mid[0][2];
      const int w0 = mid[2][0] - mid[0][0], w1 = mid[2][1] - mid[0][1], w2 = mid[2][2] - mid[0][2];
      const int dot = (u1 * w2 - u2 * w1) * dir[0] + (u2 * w0 - u0 * w2) * dir[1] + (u0 * w1 - u1 * w0) * dir[2];
      if (tri < max_t) {
        tris[3 * tri] = (int32_t)idx[0];
        tris[3 * tri + 1] = (int32_t)(dot > 0 ? idx[1] : idx[2]);
        tris[3 * tri + 2] = (int32_t)(dot > 0 ? idx[2] : idx[1]);
      }
    }
  }
}

int64_t tile_count(int64_t n) { return cdiv(n, kTile); }

int carve_iso(void* workspace, int64_t bytes, int64_t n, Workspace* w) {
  char* base = (char*)workspace;
  int64_t off = 0;
  auto take = [&](int64_t b) { const int64_t o = off; off += align_up(b, 256); return base + o; };
  const int64_t tiles = tile_count(n);
  w->mask = (uint8_t*)take(n);
  w->vloc = (uint16_t*)take(2 * n);
  w->tloc = (uint16_t*)take(2 * n);
  w->tile_sum = (int32_t*)take(8 * tiles);
  w->tile_off = (int64_t*)take(16 * tiles);
  if (workspace == nullptr || bytes < off)
    return fail(KNERF_ERR_WORKSPACE, "isosurface: workspace %lld < %lld bytes", (long long)bytes, (long long)off);
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0)
    return fail(KNERF_ERR_INVALID, "isosurface: workspace must be 256-byte aligned");
  return KNERF_OK;
}

int check_grid(int nx, int ny, int nz, Grid* g) {
  KN_CHECK_ARG(nx >= 2 && ny >= 2 && nz >= 2, "isosurface: grid %d x %d x %d, need >= 2 points per axis", nx, ny, nz);
  g->nx = nx; g->ny = ny; g->nz = nz;
  g->n = (int64_t)nx * ny * nz;
  // emit launches one thread per point in a 1-D grid of at most 2^31 - 1 blocks
  KN_CHECK_ARG(cdiv(g->n, kThreads) < (int64_t(1) << 31), "isosurface: grid of %lld points too large", (long long)g->n);
  return KNERF_OK;
}

}  // namespace
}  // namespace knerf

using namespace knerf;

extern "C" int64_t knerf_isosurface_workspace_bytes(int nx, int ny, int nz) {
  Grid g;
  if (check_grid(nx, ny, nz, &g) != KNERF_OK) return -1;
  return align_up(g.n, 256) + 2 * align_up(2 * g.n, 256) + align_up(8 * tile_count(g.n), 256) +
         align_up(16 * tile_count(g.n), 256);
}

extern "C" int knerf_isosurface_count(const float* field, int nx, int ny, int nz, float iso, int64_t* counts,
                                      void* workspace, int64_t workspace_bytes, void* stream) {
  Grid g;
  KN_TRY(check_grid(nx, ny, nz, &g));
  KN_CHECK_ARG(field && counts, "knerf_isosurface_count: null pointer");
  Workspace w;
  KN_TRY(carve_iso(workspace, workspace_bytes, g.n, &w));
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t tiles = tile_count(g.n);
  iso_count_kernel<<<(unsigned)tiles, kThreads, 0, st>>>(field, g, iso, w);
  KN_LAUNCH_CHECK();
  iso_scan_kernel<<<1, kScanThreads, 0, st>>>(w, tiles, counts);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

extern "C" int knerf_isosurface_emit(const float* field, int nx, int ny, int nz, float iso, const float* origin_host,
                                     const float* spacing_host, float* vertices, float* normals, int32_t* triangles,
                                     int64_t max_vertices, int64_t max_triangles, void* workspace,
                                     int64_t workspace_bytes, void* stream) {
  Grid g;
  KN_TRY(check_grid(nx, ny, nz, &g));
  KN_CHECK_ARG(field && origin_host && spacing_host && max_vertices >= 0 && max_triangles >= 0,
               "knerf_isosurface_emit: bad arguments");
  KN_CHECK_ARG((vertices || max_vertices == 0) && (triangles || max_triangles == 0),
               "knerf_isosurface_emit: null output with a nonzero capacity");
  if (max_vertices >= (int64_t(1) << 31))
    return fail(KNERF_ERR_UNSUPPORTED, "knerf_isosurface_emit: %lld vertices do not fit int32 triangle indices",
                (long long)max_vertices);
  Workspace w;
  KN_TRY(carve_iso(workspace, workspace_bytes, g.n, &w));
  Frame fr;
  for (int c = 0; c < 3; ++c) {
    fr.origin[c] = origin_host[c];
    fr.spacing[c] = spacing_host[c];
  }
  iso_emit_kernel<<<(unsigned)cdiv(g.n, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      field, g, iso, fr, w, vertices, normals, triangles, max_vertices, max_triangles);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}
