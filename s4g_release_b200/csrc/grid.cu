// Grid build + grid-accelerated ball query and 3-NN (see grid.cuh for the exactness argument).

#include "grid.cuh"
#include <new>

namespace s4g {

// ------------------------------------------------------------------------------------------------
// build
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
grid_desc_kernel(const float* __restrict__ points, int N, int mode, float radius, GridDesc* __restrict__ desc) {
  __shared__ float s_red[6][8];
  const int b = blockIdx.x;
  const float* X = points + (size_t)b * 3 * N;
  const float inf = __int_as_float(0x7f800000);
  float lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float v = __ldg(X + (size_t)a * N + j);
      lo[a] = fminf(lo[a], v);
      hi[a] = fmaxf(hi[a], v);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
      hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
    }
    if ((threadIdx.x & 31) == 0) {
      s_red[a][threadIdx.x >> 5] = lo[a];
      s_red[3 + a][threadIdx.x >> 5] = hi[a];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int a = 0; a < 3; ++a)
      for (int w = 0; w < 8; ++w) {
        lo[a] = fminf(lo[a], s_red[a][w]);
        hi[a] = fmaxf(hi[a], s_red[3 + a][w]);
      }
    const float ex = fmaxf(hi[0] - lo[0], 0.f), ey = fmaxf(hi[1] - lo[1], 0.f), ez = fmaxf(hi[2] - lo[2], 0.f);
    float s;
    if (mode == GRID_BALL) {
      s = radius * 1.01f;
    } else {
      const float area = fmaxf(ex * ey, fmaxf(ex * ez, ey * ez));
      s = 2.0f * sqrtf(area / (float)N);
    }
    const float ext = fmaxf(ex, fmaxf(ey, ez));
    s = fmaxf(s, fmaxf(ext * 1e-3f, 1e-12f));  // never more than 1000 cells per axis; never 0
    int dx, dy, dz;
    for (int it = 0; it < 64; ++it) {
      dx = (int)floorf(ex / s) + 1;
      dy = (int)floorf(ey / s) + 1;
      dz = (int)floorf(ez / s) + 1;
      if ((long long)dx * dy * dz <= kGridCells) break;
      s *= 1.1f;  // larger cells are always valid (only less selective)
    }
    GridDesc d;
    d.ox = lo[0]; d.oy = lo[1]; d.oz = lo[2];
    d.s = s;
    d.inv_s = 1.0f / s;
    d.dx = dx; d.dy = dy; d.dz = dz;
    desc[b] = d;
  }
}

__device__ __forceinline__ int cell_key(const GridDesc& d, float x, float y, float z) {
  const int cx = cell_coord(x, d.ox, d.inv_s, d.dx);
  const int cy = cell_coord(y, d.oy, d.inv_s, d.dy);
  const int cz = cell_coord(z, d.oz, d.inv_s, d.dz);
  return (cz * d.dy + cy) * d.dx + cx;  // x fastest: an x-row of cells is contiguous in cell order
}

__global__ void __launch_bounds__(256)
grid_count_kernel(const float* __restrict__ points, int N, const GridDesc* __restrict__ desc, int* __restrict__ count) {
  const int b = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  const float* X = points + (size_t)b * 3 * N;
  const GridDesc d = desc[b];
  const int key = cell_key(d, __ldg(X + j), __ldg(X + N + j), __ldg(X + 2 * (size_t)N + j));
  atomicAdd(count + (size_t)b * kGridCells + key, 1);
}

__global__ void __launch_bounds__(256)
grid_scatter_kernel(const float* __restrict__ points, int N, const GridDesc* __restrict__ desc,
                    const int* __restrict__ start, int* __restrict__ cursor, float4* __restrict__ sorted) {
  const int b = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  const float* X = points + (size_t)b * 3 * N;
  const GridDesc d = desc[b];
  const float x = __ldg(X + j), y = __ldg(X + N + j), z = __ldg(X + 2 * (size_t)N + j);
  const size_t cell = (size_t)b * kGridCells + cell_key(d, x, y, z);
  const int slot = start[cell] + atomicAdd(cursor + cell, 1);
  sorted[slot] = make_float4(x, y, z, __int_as_float(j));  // start[] is a global prefix: slot is batch-global
}

static size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

// ---- exclusive prefix sum of the cell counts (hand-written: no library kernel on the path) ----
// scan_block_kernel: each block scans kScanTile consecutive items (4 per thread) and writes its total;
// scan_sums_kernel: one block scans the block totals; scan_add_kernel adds them back.
constexpr int kScanThreads = 1024;
constexpr int kScanTile = kScanThreads * 4;

__device__ __forceinline__ int scan_block_exclusive(int v, int* s_warp, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int w = s_warp[lane];
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    s_warp[lane] = wi - w;
    if (lane == 31) s_warp[32] = wi;
  }
  __syncthreads();
  total = s_warp[32];
  const int res = s_warp[warp] + incl - v;
  __syncthreads();
  return res;
}

__global__ void __launch_bounds__(kScanThreads) scan_block_kernel(const int* __restrict__ in, int n, int* __restrict__ out,
                                                                  int* __restrict__ sums) {
  __shared__ int s_warp[33];
  const int base = blockIdx.x * kScanTile + threadIdx.x * 4;
  int v[4], t = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    v[k] = base + k < n ? in[base + k] : 0;
    t += v[k];
  }
  int total;
  int run = scan_block_exclusive(t, s_warp, total);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (base + k < n) out[base + k] = run;
    run += v[k];
  }
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanThreads) scan_sums_kernel(int* __restrict__ sums, int n) {
  __shared__ int s_warp[33];
  int carry = 0;
  for (int base = 0; base < n; base += kScanThreads) {
    const int i = base + threadIdx.x;
    const int v = i < n ? sums[i] : 0;
    int total;
    const int ex = scan_block_exclusive(v, s_warp, total);
    if (i < n) sums[i] = carry + ex;
    carry += total;
  }
}

__global__ void __launch_bounds__(kScanThreads) scan_add_kernel(int* __restrict__ out, int n, const int* __restrict__ sums) {
  const int add = sums[blockIdx.x];
  const int base = blockIdx.x * kScanTile + threadIdx.x * 4;
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (base + k < n) out[base + k] += add;
}

int grid_build(const float* points, int B, int N, int mode, float radius, Grid* g, cudaStream_t stream) {
  const size_t cells = (size_t)B * kGridCells;
  const int scan_n = (int)cells + 1;
  const int scan_blocks = (scan_n + kScanTile - 1) / kScanTile;
  const size_t scan_tmp = sizeof(int) * (size_t)scan_blocks;
  const size_t o_desc = 0;
  const size_t o_count = o_desc + align_up(sizeof(GridDesc) * B);
  const size_t o_cursor = o_count + align_up(sizeof(int) * (cells + 1));
  const size_t o_start = o_cursor + align_up(sizeof(int) * cells);
  const size_t o_sorted = o_start + align_up(sizeof(int) * (cells + 1));
  const size_t o_tmp = o_sorted + align_up(sizeof(float4) * (size_t)B * N);
  const size_t total = o_tmp + align_up(scan_tmp);
  // keep freed blocks in the stream-ordered pool instead of returning them to the OS — once PER DEVICE (one process may
  // drive several GPUs, e.g. nn.DataParallel replicas); a racing duplicate call from another thread is harmless
  static bool pool_ready[64] = {};
  int dev = 0;
  S4G_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && !pool_ready[dev]) {
    cudaMemPool_t pool;
    S4G_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    uint64_t keep = ~0ull;
    S4G_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    pool_ready[dev] = true;
  }
  uint8_t* arena = nullptr;
  S4G_CUDA(cudaMallocAsync((void**)&arena, total, stream));
  g->arena = arena;
  g->desc = reinterpret_cast<GridDesc*>(arena + o_desc);
  int* count = reinterpret_cast<int*>(arena + o_count);
  int* cursor = reinterpret_cast<int*>(arena + o_cursor);
  g->start = reinterpret_cast<int*>(arena + o_start);
  g->sorted = reinterpret_cast<float4*>(arena + o_sorted);
  g->B = B;
  g->N = N;
  // count and cursor are adjacent: one memset clears both
  S4G_CUDA(cudaMemsetAsync(count, 0, o_start - o_count, stream));
  grid_desc_kernel<<<B, 256, 0, stream>>>(points, N, mode, radius, g->desc);
  S4G_LAUNCH_CHECK("grid_desc");
  dim3 grid((N + 255) / 256, B);
  grid_count_kernel<<<grid, 256, 0, stream>>>(points, N, g->desc, count);
  S4G_LAUNCH_CHECK("grid_count");
  int* sums = reinterpret_cast<int*>(arena + o_tmp);
  scan_block_kernel<<<scan_blocks, kScanThreads, 0, stream>>>(count, scan_n, g->start, sums);
  S4G_LAUNCH_CHECK("grid_scan");
  if (scan_blocks > 1) {
    scan_sums_kernel<<<1, kScanThreads, 0, stream>>>(sums, scan_blocks);
    S4G_LAUNCH_CHECK("grid_scan_sums");
    scan_add_kernel<<<scan_blocks, kScanThreads, 0, stream>>>(g->start, scan_n, sums);
    S4G_LAUNCH_CHECK("grid_scan_add");
  }
  grid_scatter_kernel<<<grid, 256, 0, stream>>>(points, N, g->desc, g->start, cursor, g->sorted);
  S4G_LAUNCH_CHECK("grid_scatter");
  return S4G_OK;
}

int grid_free(Grid* g, cudaStream_t stream) {
  if (g->arena) S4G_CUDA(cudaFreeAsync(g->arena, stream));
  g->arena = nullptr;
  return S4G_OK;
}

// ------------------------------------------------------------------------------------------------
// ball query on the grid: one warp per centroid
// ------------------------------------------------------------------------------------------------
constexpr int kBqgWarps = 8;
constexpr int kBqgCap = 256;  // hits buffered per centroid before falling back to the exact linear scan

__device__ __forceinline__ void warp_sort_ascending(int* buf, int n, int lane) {  // n = power of two
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < n; i += 32) {
        const int p = i ^ j;
        if (p > i) {
          const int a = buf[i], b = buf[p];
          const bool up = (i & k) == 0;
          if ((a > b) == up) { buf[i] = b; buf[p] = a; }
        }
      }
      __syncwarp();
    }
  }
}

template <typename IndexT>
__global__ void __launch_bounds__(kBqgWarps * 32)
ball_query_grid_kernel(const float* __restrict__ points, const float* __restrict__ centroids, int N, int M, float r2,
                       int K, const GridDesc* __restrict__ desc, const int* __restrict__ start,
                       const float4* __restrict__ sorted, IndexT* __restrict__ index, IndexT* __restrict__ count) {
  __shared__ int s_hits[kBqgWarps][kBqgCap];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int m = blockIdx.x * kBqgWarps + warp;
  if (m >= M) return;
  const float* CX = centroids + (size_t)b * 3 * M;
  const float cx = __ldg(CX + m), cy = __ldg(CX + M + m), cz = __ldg(CX + 2 * (size_t)M + m);
  const GridDesc d = desc[b];
  const int gx = cell_coord(cx, d.ox, d.inv_s, d.dx);
  const int gy = cell_coord(cy, d.oy, d.inv_s, d.dy);
  const int gz = cell_coord(cz, d.oz, d.inv_s, d.dz);
  const int x0 = max(gx - 1, 0), x1 = min(gx + 1, d.dx - 1);
  const int* st = start + (size_t)b * kGridCells;
  int* hits = s_hits[warp];
  const unsigned lt = (1u << lane) - 1u;
  int H = 0;
  for (int zz = max(gz - 1, 0); zz <= min(gz + 1, d.dz - 1); ++zz) {
    for (int yy = max(gy - 1, 0); yy <= min(gy + 1, d.dy - 1); ++yy) {
      const int row = (zz * d.dy + yy) * d.dx;
      const int a = __ldg(st + row + x0), e = __ldg(st + row + x1 + 1);  // contiguous x-row of cells
      for (int base = a; base < e; base += 32) {
        const int i = base + lane;
        const bool v = i < e;
        float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
        if (v) p = __ldg(sorted + i);
        const float dd = sqdist(__fsub_rn(p.x, cx), __fsub_rn(p.y, cy), __fsub_rn(p.z, cz));
        const bool hit = v && (dd < r2);
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (bal) {
          const int pos = H + __popc(bal & lt);
          if (hit && pos < kBqgCap) hits[pos] = __float_as_int(p.w);
          H += __popc(bal);
        }
      }
    }
  }
  IndexT* out = index + ((size_t)b * M + m) * K;
  if (H > kBqgCap) {
    // more candidates than the buffer holds: exact linear scan in index order (rare: degenerate clouds)
    const float* X = points + (size_t)b * 3 * N;
    int cnt = 0, first = 0;
    for (int base = 0; base < N && cnt < K; base += 32) {
      const int j = base + lane;
      const bool v = j < N;
      const float x = v ? __ldg(X + j) : 0.f, y = v ? __ldg(X + N + j) : 0.f, z = v ? __ldg(X + 2 * (size_t)N + j) : 0.f;
      const float dd = sqdist(__fsub_rn(x, cx), __fsub_rn(y, cy), __fsub_rn(z, cz));
      const bool hit = v && (dd < r2);
      const unsigned bal = __ballot_sync(0xffffffffu, hit);
      if (bal) {
        const int pos = cnt + __popc(bal & lt);
        if (hit && pos < K) out[pos] = (IndexT)j;
        if (cnt == 0) first = base + __ffs(bal) - 1;
        cnt = min(cnt + __popc(bal), K);
      }
    }
    for (int k = cnt + lane; k < K; k += 32) out[k] = (IndexT)first;
    if (lane == 0 && count != nullptr) count[(size_t)b * M + m] = (IndexT)cnt;
    return;
  }
  __syncwarp();
  int n2 = 32;
  while (n2 < H) n2 <<= 1;
  for (int i = H + lane; i < n2; i += 32) hits[i] = 0x7fffffff;
  __syncwarp();
  if (H > 1) warp_sort_ascending(hits, n2, lane);
  const int cnt = min(H, K);
  const int first = (H > 0) ? hits[0] : 0;
  for (int k = lane; k < K; k += 32) out[k] = (IndexT)((k < cnt) ? hits[k] : first);
  if (lane == 0 && count != nullptr) count[(size_t)b * M + m] = (IndexT)cnt;
}

template <typename IndexT>
int ball_query_grid(const float* points, const float* centroids, int B, int N, int M, float radius, int K,
                    IndexT* index, IndexT* count, cudaStream_t stream) {
  Grid g = {};
  int rc = grid_build(points, B, N, GRID_BALL, radius, &g, stream);
  if (rc != S4G_OK) return rc;
  const float r2 = radius * radius;
  dim3 grid((M + kBqgWarps - 1) / kBqgWarps, B);
  ball_query_grid_kernel<IndexT><<<grid, kBqgWarps * 32, 0, stream>>>(points, centroids, N, M, r2, K, g.desc, g.start,
                                                                    g.sorted, index, count);
  S4G_LAUNCH_CHECK("ball_query_grid");
  return grid_free(&g, stream);
}

template int ball_query_grid<int64_t>(const float*, const float*, int, int, int, float, int, int64_t*, int64_t*,
                                      cudaStream_t);
template int ball_query_grid<int32_t>(const float*, const float*, int, int, int, float, int, int32_t*, int32_t*,
                                      cudaStream_t);

// ------------------------------------------------------------------------------------------------
// 3-NN on the grid: thread per query over the 3x3x3 block; unresolved queries -> exact warp-per-query pass
// ------------------------------------------------------------------------------------------------
struct Top3 {
  float d0, d1, d2;
  int i0, i1, i2;
};

// ordering of the reference's insertion over keys in index order: (d2, index) lexicographic
__device__ __forceinline__ bool closer(float d, int j, float dk, int ik) { return d < dk || (d == dk && j < ik); }

__device__ __forceinline__ void top3_insert(Top3& t, float d, int j) {
  if (closer(d, j, t.d2, t.i2)) {
    if (closer(d, j, t.d1, t.i1)) {
      t.d2 = t.d1; t.i2 = t.i1;
      if (closer(d, j, t.d0, t.i0)) { t.d1 = t.d0; t.i1 = t.i0; t.d0 = d; t.i0 = j; }
      else { t.d1 = d; t.i1 = j; }
    } else { t.d2 = d; t.i2 = j; }
  }
}

// output: MODE 0 -> int64 index + squared distance (pn2_ext.point_search); MODE 1 -> int32 index + weights.
// Slots without a key below +inf (they hold +inf / 0x7fffffff, or a key kept on a tie at +inf) become the reference's
// leftovers first; MODE 1 then computes the weights from those distances and writes index 0 for the reference's -1,
// whose weight is 1/inf = 0, so every index it writes is a valid key row.
template <int MODE>
__device__ __forceinline__ void top3_store(Top3 t, size_t q, void* index, float* out) {
  three_nn_reference_tail(t.d0, t.d1, t.d2, t.i0, t.i1, t.i2, __int_as_float(0x7f800000));
  if (MODE == 0) {
    int64_t* oi = reinterpret_cast<int64_t*>(index) + q * 3;
    oi[0] = t.i0; oi[1] = t.i1; oi[2] = t.i2;
    out[q * 3 + 0] = t.d0; out[q * 3 + 1] = t.d1; out[q * 3 + 2] = t.d2;
  } else {
    int* oi = reinterpret_cast<int*>(index) + q * 3;
    oi[0] = max(t.i0, 0); oi[1] = max(t.i1, 0); oi[2] = max(t.i2, 0);
    const float v0 = __fdiv_rn(1.0f, fmaxf(t.d0, 1e-10f));
    const float v1 = __fdiv_rn(1.0f, fmaxf(t.d1, 1e-10f));
    const float v2 = __fdiv_rn(1.0f, fmaxf(t.d2, 1e-10f));
    const float norm = __fadd_rn(__fadd_rn(v0, v1), v2);
    out[q * 3 + 0] = __fdiv_rn(v0, norm); out[q * 3 + 1] = __fdiv_rn(v1, norm); out[q * 3 + 2] = __fdiv_rn(v2, norm);
  }
}

template <int MODE>
__global__ void __launch_bounds__(256)
three_nn_grid_kernel(const float* __restrict__ query, int Nq, const GridDesc* __restrict__ desc,
                     const int* __restrict__ start, const float4* __restrict__ sorted, void* __restrict__ index,
                     float* __restrict__ out, int* __restrict__ pending, int* __restrict__ n_pending) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Nq) return;
  const float* Q = query + (size_t)b * 3 * Nq;
  const float qx = __ldg(Q + i), qy = __ldg(Q + Nq + i), qz = __ldg(Q + 2 * (size_t)Nq + i);
  const GridDesc d = desc[b];
  const int gx = cell_coord(qx, d.ox, d.inv_s, d.dx);
  const int gy = cell_coord(qy, d.oy, d.inv_s, d.dy);
  const int gz = cell_coord(qz, d.oz, d.inv_s, d.dz);
  const int x0 = max(gx - 1, 0), x1 = min(gx + 1, d.dx - 1);
  const int* st = start + (size_t)b * kGridCells;
  const float inf = __int_as_float(0x7f800000);
  Top3 t = {inf, inf, inf, 0x7fffffff, 0x7fffffff, 0x7fffffff};
  for (int zz = max(gz - 1, 0); zz <= min(gz + 1, d.dz - 1); ++zz) {
    for (int yy = max(gy - 1, 0); yy <= min(gy + 1, d.dy - 1); ++yy) {
      const int row = (zz * d.dy + yy) * d.dx;
      const int a = __ldg(st + row + x0), e = __ldg(st + row + x1 + 1);
      for (int k = a; k < e; ++k) {
        const float4 p = __ldg(sorted + k);
        // the reference computes query - key (interpolate_kernel.cu:62)
        const float dd = sqdist(__fsub_rn(qx, p.x), __fsub_rn(qy, p.y), __fsub_rn(qz, p.z));
        top3_insert(t, dd, __float_as_int(p.w));
      }
    }
  }
  // every key outside the block is farther than 0.999 * cell edge: the block result is exact iff the
  // third distance is below that bound (strictly, so no outside key can even tie)
  const float lim = 0.999f * d.s;
  const size_t q = (size_t)b * Nq + i;
  if (t.d2 < lim * lim) top3_store<MODE>(t, q, index, out);
  else pending[atomicAdd(n_pending, 1)] = (int)q;
}

// exact pass for the unresolved queries: one warp per query, lanes stride the keys in index order
template <int MODE>
__global__ void __launch_bounds__(256)
three_nn_pending_kernel(const float* __restrict__ query, const float* __restrict__ key, int Nq, int Nk,
                        const int* __restrict__ pending, const int* __restrict__ n_pending, void* __restrict__ index,
                        float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int total = *n_pending;
  const float inf = __int_as_float(0x7f800000);
  for (int w = blockIdx.x * 8 + (threadIdx.x >> 5); w < total; w += gridDim.x * 8) {
    const int q = pending[w];
    const int b = q / Nq, i = q - b * Nq;
    const float* Q = query + (size_t)b * 3 * Nq;
    const float* KX = key + (size_t)b * 3 * Nk;
    const float qx = __ldg(Q + i), qy = __ldg(Q + Nq + i), qz = __ldg(Q + 2 * (size_t)Nq + i);
    Top3 t = {inf, inf, inf, 0x7fffffff, 0x7fffffff, 0x7fffffff};
    for (int j = lane; j < Nk; j += 32) {
      const float dd = sqdist(__fsub_rn(qx, __ldg(KX + j)), __fsub_rn(qy, __ldg(KX + Nk + j)),
                              __fsub_rn(qz, __ldg(KX + 2 * (size_t)Nk + j)));
      top3_insert(t, dd, j);
    }
    // merge the 32 per-lane lists: three rounds of warp arg-min on (d, index)
    Top3 r = {inf, inf, inf, 0x7fffffff, 0x7fffffff, 0x7fffffff};
    for (int round = 0; round < 3; ++round) {
      float bd = t.d0;
      int bi = t.i0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(0xffffffffu, bd, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (closer(od, oi, bd, bi)) { bd = od; bi = oi; }
      }
      if (round == 0) { r.d0 = bd; r.i0 = bi; }
      else if (round == 1) { r.d1 = bd; r.i1 = bi; }
      else { r.d2 = bd; r.i2 = bi; }
      if (t.i0 == bi && t.d0 == bd) {  // the winning lane pops its head
        t.d0 = t.d1; t.i0 = t.i1; t.d1 = t.d2; t.i1 = t.i2; t.d2 = inf; t.i2 = 0x7fffffff;
      }
    }
    if (lane == 0) top3_store<MODE>(r, (size_t)q, index, out);
  }
}

template <int MODE>
int three_nn_grid(const float* query, const float* key, int B, int Nq, int Nk, void* index, float* out,
                  cudaStream_t stream) {
  Grid g = {};
  int rc = grid_build(key, B, Nk, GRID_KNN, 0.f, &g, stream);
  if (rc != S4G_OK) return rc;
  int* pending = nullptr;
  S4G_CUDA(cudaMallocAsync((void**)&pending, sizeof(int) * ((size_t)B * Nq + 1), stream));
  int* n_pending = pending + (size_t)B * Nq;
  S4G_CUDA(cudaMemsetAsync(n_pending, 0, sizeof(int), stream));
  dim3 grid((Nq + 255) / 256, B);
  three_nn_grid_kernel<MODE><<<grid, 256, 0, stream>>>(query, Nq, g.desc, g.start, g.sorted, index, out, pending,
                                                       n_pending);
  S4G_LAUNCH_CHECK("three_nn_grid");
  three_nn_pending_kernel<MODE><<<num_sms() * 4, 256, 0, stream>>>(query, key, Nq, Nk, pending, n_pending, index, out);
  S4G_LAUNCH_CHECK("three_nn_grid");
  S4G_CUDA(cudaFreeAsync(pending, stream));
  return grid_free(&g, stream);
}

template int three_nn_grid<0>(const float*, const float*, int, int, int, void*, float*, cudaStream_t);
template int three_nn_grid<1>(const float*, const float*, int, int, int, void*, float*, cudaStream_t);

}  // namespace s4g

// ------------------------------------------------------------------------------------------------
// Ball query in two calls: the index over the points only needs the cloud, so a caller can build it on another stream
// while the centroids are still being sampled (engine.py runs it beside the first level's farthest point sampling).
// ------------------------------------------------------------------------------------------------
struct s4g_ball_grid {
  s4g::Grid grid;
  float radius;
};

extern "C" int s4g_ball_query_uses_grid(int N, int K, float radius) {
  return (N >= s4g::kGridBallMinPoints && K <= s4g::kGridBallMaxK && radius > 0.f) ? 1 : 0;
}

extern "C" s4g_ball_grid* s4g_ball_grid_build_f32(const float* points, int B, int N, float radius, void* stream) {
  if (!points || B <= 0 || B > 65535 || N < 1 || !(radius > 0.f)) {
    s4g::set_error(S4G_E_ARG, "ball_grid_build: bad cloud or radius");
    return nullptr;
  }
  s4g_ball_grid* g = new (std::nothrow) s4g_ball_grid();
  if (!g) return nullptr;
  g->radius = radius;
  if (s4g::grid_build(points, B, N, s4g::GRID_BALL, radius, &g->grid, (cudaStream_t)stream) != S4G_OK) {
    delete g;
    return nullptr;
  }
  return g;
}

// same result as s4g_ball_query_f32_i32 on the cloud the grid was built from; `stream` must be ordered after the build
extern "C" int s4g_ball_query_with_grid_f32_i32(const s4g_ball_grid* g, const float* points, const float* centroids, int M,
                                                int K, int32_t* index, int32_t* count, void* stream) {
  S4G_CHECK_ARG(g && points && centroids && index, "ball_query_with_grid: null pointer");
  S4G_CHECK_ARG(M > 0 && K > 0 && K <= s4g::kGridBallMaxK, "ball_query_with_grid: bad shape");
  const float r2 = g->radius * g->radius;
  dim3 grid((M + s4g::kBqgWarps - 1) / s4g::kBqgWarps, g->grid.B);
  s4g::ball_query_grid_kernel<int32_t><<<grid, s4g::kBqgWarps * 32, 0, (cudaStream_t)stream>>>(
      points, centroids, g->grid.N, M, r2, K, g->grid.desc, g->grid.start, g->grid.sorted, index, count);
  S4G_LAUNCH_CHECK("ball_query_grid");
  return S4G_OK;
}

// releases the index (stream-ordered: after the queries issued on `stream`)
extern "C" int s4g_ball_grid_free(s4g_ball_grid* g, void* stream) {
  if (!g) return S4G_OK;
  const int rc = s4g::grid_free(&g->grid, (cudaStream_t)stream);
  delete g;
  return rc;
}
