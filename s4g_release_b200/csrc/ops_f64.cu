// fp64 instantiation of the seven pn2_ext operators.  The reference dispatches every kernel over float AND
// double (AT_DISPATCH_FLOATING_TYPES: csrc/sampling_kernel.cu:21, ball_query_kernel.cu:116,
// grouping_kernel.cu:137, interpolate_kernel.cu:118,222,327); the model itself runs fp32, so these are the
// completeness path of the drop-in boundary, written for exactness first: plain one-CTA-per-cloud /
// one-warp-per-centroid kernels, same selection rules as the fp32 kernels, distances in the order the
// reference's double SASS uses (DMUL dy*dy ; DFMA dx*dx + . ; DFMA dz*dz + .).
#include "common.cuh"

namespace s4g {

__device__ __forceinline__ double sqdist64(double dx, double dy, double dz) {
  return __fma_rn(dz, dz, __fma_rn(dx, dx, __dmul_rn(dy, dy)));
}

constexpr int kFps64Threads = 1024;

// Farthest point sampling (sampling_kernel.cu:49-119).  The reference's winner among equal maxima is the
// point minimising (bitreverse_{log2 BLOCK}(j mod BLOCK), j), BLOCK = its own block size for this N
// (derivation: oracle/pn2_oracle_body.inc, farthest_point_sample_keyed); a maximum of 0 repeats the previous index.
// temp: running minimum distance, in shared memory when the cloud fits, else in the caller-provided workspace.
__global__ void __launch_bounds__(kFps64Threads)
fps64_kernel(const double* __restrict__ points, int N, int M, int ref_block_log2, double* __restrict__ temp_g,
             int temp_in_smem, int64_t* __restrict__ index) {
  extern __shared__ double s_temp[];
  __shared__ double s_d[32];
  __shared__ unsigned long long s_k[32];
  __shared__ int s_cur;
  const int b = blockIdx.x;
  const double* X = points + (size_t)b * 3 * N;
  const double* Y = X + N;
  const double* Z = Y + N;
  double* temp = temp_in_smem ? s_temp : temp_g + (size_t)b * N;
  int64_t* out = index + (size_t)b * M;
  const int L = ref_block_log2;
  const unsigned mask = (1u << L) - 1u;
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  for (int j = threadIdx.x; j < N; j += kFps64Threads) temp[j] = inf;
  if (threadIdx.x == 0) out[0] = 0;
  int cur = 0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = 1; i < M; ++i) {
    const double x1 = X[cur], y1 = Y[cur], z1 = Z[cur];
    double best = 0.0;
    unsigned long long best_k = ~0ull;  // low 32 bits = the index; (0, ~0) stands for "repeat cur"
    for (int j = threadIdx.x; j < N; j += kFps64Threads) {
      double d = sqdist64(X[j] - x1, Y[j] - y1, Z[j] - z1);
      const double t = temp[j];
      if (d < t) temp[j] = d; else d = t;
      const unsigned long long k = ((unsigned long long)(__brev((unsigned)j & mask) >> (32 - L)) << 32) | (unsigned)j;
      if (d > best || (d == best && d > 0.0 && k < best_k)) { best = d; best_k = k; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, best, o);
      const unsigned long long ok = __shfl_xor_sync(0xffffffffu, best_k, o);
      if (od > best || (od == best && ok < best_k)) { best = od; best_k = ok; }
    }
    if (lane == 0) { s_d[warp] = best; s_k[warp] = best_k; }
    __syncthreads();
    if (warp == 0) {
      best = s_d[lane];
      best_k = s_k[lane];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, best, o);
        const unsigned long long ok = __shfl_xor_sync(0xffffffffu, best_k, o);
        if (od > best || (od == best && ok < best_k)) { best = od; best_k = ok; }
      }
      if (lane == 0) {
        const int nxt = best > 0.0 ? (int)(unsigned)(best_k & 0xffffffffull) : cur;
        s_cur = nxt;
        out[i] = nxt;
      }
    }
    __syncthreads();
    cur = s_cur;
  }
}

// Ball query (ball_query_kernel.cu:33-76): one warp per centroid scans the cloud 32 points at a time in
// ascending order; hits are placed by ballot + prefix count, the first hit pre-fills all K slots, the scan
// stops at K hits.  index zero-initialised when there is no hit (:109).
__global__ void __launch_bounds__(256)
ball_query64_kernel(const double* __restrict__ points, const double* __restrict__ centroids, int N, int M, double r2,
                    int K, int64_t* __restrict__ index, int64_t* __restrict__ count) {
  const int b = blockIdx.y;
  const int m = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (m >= M) return;
  const double* X = points + (size_t)b * 3 * N;
  const double* Y = X + N;
  const double* Z = Y + N;
  const double* C = centroids + (size_t)b * 3 * M;
  const double x1 = C[m], y1 = C[M + m], z1 = C[2 * M + m];
  int64_t* idx = index + ((size_t)b * M + m) * K;
  int cnt = 0;
  for (int base = 0; base < N && cnt < K; base += 32) {
    const int j = base + lane;
    bool hit = false;
    if (j < N) hit = sqdist64(X[j] - x1, Y[j] - y1, Z[j] - z1) < r2;
    const unsigned bal = __ballot_sync(0xffffffffu, hit);
    if (bal == 0u) continue;
    if (cnt == 0) {
      const int first = base + __ffs(bal) - 1;
      for (int k = lane; k < K; k += 32) idx[k] = first;
      __syncwarp();
    }
    const int pos = cnt + __popc(bal & ((1u << lane) - 1u));
    if (hit && pos < K && pos > 0) idx[pos] = j;
    cnt += __popc(bal);
  }
  if (cnt == 0)
    for (int k = lane; k < K; k += 32) idx[k] = 0;
  if (lane == 0) count[(size_t)b * M + m] = cnt < K ? cnt : K;
}

__global__ void __launch_bounds__(256)
group_forward64_kernel(const double* __restrict__ input, const int64_t* __restrict__ index, int C, int N, int MK,
                       double* __restrict__ out) {
  const int b = blockIdx.y;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= MK) return;
  const int64_t j = index[(size_t)b * MK + q];
  const double* in = input + (size_t)b * C * N + j;
  double* o = out + (size_t)b * C * MK + q;
  for (int c = 0; c < C; ++c) o[(size_t)c * MK] = __ldg(in + (size_t)c * N);
}

__global__ void __launch_bounds__(256)
group_backward64_kernel(const double* __restrict__ grad_out, const int64_t* __restrict__ index, int C, int N, int MK,
                        double* __restrict__ grad_in) {
  const int b = blockIdx.y;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= MK) return;
  const int64_t j = index[(size_t)b * MK + q];
  double* gi = grad_in + (size_t)b * C * N + j;
  const double* go = grad_out + (size_t)b * C * MK + q;
  for (int c = 0; c < C; ++c) atomicAdd(gi + (size_t)c * N, __ldg(go + (size_t)c * MK));
}

// 3-NN (interpolate_kernel.cu:33-81): one thread per query, keys staged through shared memory; strict '<'
// insertion in key order.  The reference starts from {1e40, 0, 0} / {-1, 0, 0}: the same state as this all-1e40 start
// once two keys are closer than 1e40; three_nn_reference_tail restores the reference's slots when fewer are.
constexpr int kNn64Tile = 1024;
__global__ void __launch_bounds__(256)
point_search64_kernel(const double* __restrict__ query, const double* __restrict__ key, int Nq, int Nk,
                      int64_t* __restrict__ index, double* __restrict__ distance) {
  __shared__ double s_x[kNn64Tile], s_y[kNn64Tile], s_z[kNn64Tile];
  const int b = blockIdx.y;
  const int i = blockIdx.x * 256 + threadIdx.x;
  const bool valid = i < Nq;
  const double* Q = query + (size_t)b * 3 * Nq;
  const double* KX = key + (size_t)b * 3 * Nk;
  const double* KY = KX + Nk;
  const double* KZ = KY + Nk;
  const int iq = valid ? i : Nq - 1;
  const double x1 = Q[iq], y1 = Q[Nq + iq], z1 = Q[2 * Nq + iq];
  double d0 = 1e40, d1 = 1e40, d2 = 1e40;
  int i0 = -1, i1 = -1, i2 = -1;
  for (int base = 0; base < Nk; base += kNn64Tile) {
    const int n = min(kNn64Tile, Nk - base);
    __syncthreads();
    for (int k = threadIdx.x; k < n; k += 256) { s_x[k] = KX[base + k]; s_y[k] = KY[base + k]; s_z[k] = KZ[base + k]; }
    __syncthreads();
    for (int k = 0; k < n; ++k) {
      const double d = sqdist64(x1 - s_x[k], y1 - s_y[k], z1 - s_z[k]);
      if (d < d2) {
        const int j = base + k;
        if (d < d1) {
          d2 = d1; i2 = i1;
          if (d < d0) { d1 = d0; i1 = i0; d0 = d; i0 = j; }
          else { d1 = d; i1 = j; }
        } else { d2 = d; i2 = j; }
      }
    }
  }
  if (valid) {
    three_nn_reference_tail(d0, d1, d2, i0, i1, i2, 1e40);
    int64_t* oi = index + ((size_t)b * Nq + i) * 3;
    double* od = distance + ((size_t)b * Nq + i) * 3;
    oi[0] = i0; oi[1] = i1; oi[2] = i2;
    od[0] = d0; od[1] = d1; od[2] = d2;
  }
}

__global__ void __launch_bounds__(256)
interpolate_forward64_kernel(const double* __restrict__ input, const int64_t* __restrict__ index,
                             const double* __restrict__ weight, int C, int Nk, int Nq, double* __restrict__ out) {
  const int b = blockIdx.y;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= Nq) return;
  const int64_t* idx = index + ((size_t)b * Nq + n) * 3;
  const double* w = weight + ((size_t)b * Nq + n) * 3;
  const int64_t j0 = idx[0], j1 = idx[1], j2 = idx[2];
  const double w0 = w[0], w1 = w[1], w2 = w[2];
  const double* in = input + (size_t)b * C * Nk;
  double* o = out + (size_t)b * C * Nq + n;
  for (int c = 0; c < C; ++c) {
    const double* ic = in + (size_t)c * Nk;
    double v = __fma_rn(__ldg(ic + j0), w0, 0.0);
    v = __fma_rn(__ldg(ic + j1), w1, v);
    v = __fma_rn(__ldg(ic + j2), w2, v);
    o[(size_t)c * Nq] = v;
  }
}

__global__ void __launch_bounds__(256)
interpolate_backward64_kernel(const double* __restrict__ grad_out, const int64_t* __restrict__ index,
                              const double* __restrict__ weight, int C, int Nk, int Nq, double* __restrict__ grad_in) {
  const int b = blockIdx.y;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= Nq) return;
  const int64_t* idx = index + ((size_t)b * Nq + n) * 3;
  const double* w = weight + ((size_t)b * Nq + n) * 3;
  const int64_t j0 = idx[0], j1 = idx[1], j2 = idx[2];
  const double w0 = w[0], w1 = w[1], w2 = w[2];
  double* gi = grad_in + (size_t)b * C * Nk;
  const double* go = grad_out + (size_t)b * C * Nq + n;
  for (int c = 0; c < C; ++c) {
    const double g = __ldg(go + (size_t)c * Nq);
    double* gc = gi + (size_t)c * Nk;
    atomicAdd(gc + j0, __dmul_rn(g, w0));
    atomicAdd(gc + j1, __dmul_rn(g, w1));
    atomicAdd(gc + j2, __dmul_rn(g, w2));
  }
}

}  // namespace s4g

extern "C" size_t s4g_farthest_point_sample_f64_workspace(int B, int N) {
  const size_t per_cloud = sizeof(double) * (size_t)N;
  return per_cloud <= 200 * 1024 ? 0 : per_cloud * (size_t)B;
}

extern "C" int s4g_farthest_point_sample_f64(const double* points, int B, int N, int M, int64_t* index, void* workspace,
                                             size_t workspace_bytes, void* stream) {
  S4G_CHECK_ARG(points && index, "farthest_point_sample: null pointer");
  S4G_CHECK_ARG(M > 0, "farthest_point_sample: num_centroids <= 0");          // sampling_kernel.cu:138
  S4G_CHECK_ARG(N >= M, "farthest_point_sample: num_points < num_centroids");  // :139
  S4G_CHECK_ARG(B >= 0, "farthest_point_sample: bad batch");
  if (B == 0) return S4G_OK;
  const size_t need = s4g_farthest_point_sample_f64_workspace(B, N);
  S4G_CHECK_ARG(workspace_bytes >= need && (need == 0 || workspace), "farthest_point_sample: workspace too small");
  int block = 16, L = 4;  // the reference's block size for this N (sampling_kernel.cu:34-42,150-167)
  while (block < N && block < 512) { block <<= 1; ++L; }
  const size_t smem = need == 0 ? sizeof(double) * (size_t)N : 0;
  static bool attr_set[64] = {};
  if (s4g::first_use_on_device(attr_set)) {
    S4G_CUDA(cudaFuncSetAttribute(s4g::fps64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  s4g::fps64_kernel<<<B, s4g::kFps64Threads, smem, (cudaStream_t)stream>>>(points, N, M, L, (double*)workspace,
                                                                          need == 0 ? 1 : 0, index);
  S4G_LAUNCH_CHECK("farthest_point_sample_f64");
  return S4G_OK;
}

extern "C" int s4g_ball_query_f64(const double* points, const double* centroids, int B, int N, int M, double radius, int K,
                                  int64_t* index, int64_t* count, void* stream) {
  S4G_CHECK_ARG(points && centroids && index && count, "ball_query: null pointer");
  S4G_CHECK_ARG(B >= 0 && N > 0 && M > 0 && K > 0, "ball_query: bad shape");
  S4G_CHECK_ARG(B <= 65535, "ball_query: batch too large for one launch");
  if (B == 0) return S4G_OK;
  dim3 grid((M + 7) / 8, B);
  s4g::ball_query64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(points, centroids, N, M, radius * radius, K, index,
                                                                   count);
  S4G_LAUNCH_CHECK("ball_query_f64");
  return S4G_OK;
}

extern "C" int s4g_group_points_forward_f64(const double* input, const int64_t* index, int B, int C, int N, int M, int K,
                                            double* out, void* stream) {
  S4G_CHECK_ARG(input && index && out, "group_points_forward: null pointer");
  S4G_CHECK_ARG(B >= 0 && C > 0 && N > 0 && M > 0 && K > 0, "group_points_forward: bad shape");
  S4G_CHECK_ARG(B <= 65535, "group_points_forward: batch too large for one launch");
  S4G_CHECK_ARG((long long)M * K < (1ll << 31), "group_points_forward: M*K too large");
  if (B == 0) return S4G_OK;
  const int MK = M * K;
  dim3 grid((MK + 255) / 256, B);
  s4g::group_forward64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(input, index, C, N, MK, out);
  S4G_LAUNCH_CHECK("group_points_forward_f64");
  return S4G_OK;
}

extern "C" int s4g_group_points_backward_f64(const double* grad_out, const int64_t* index, int B, int C, int N, int M,
                                             int K, double* grad_in, void* stream) {
  S4G_CHECK_ARG(grad_out && index && grad_in, "group_points_backward: null pointer");
  S4G_CHECK_ARG(B >= 0 && C > 0 && N > 0 && M > 0 && K > 0, "group_points_backward: bad shape");
  S4G_CHECK_ARG(B <= 65535, "group_points_backward: batch too large for one launch");
  S4G_CHECK_ARG((long long)M * K < (1ll << 31), "group_points_backward: M*K too large");
  if (B == 0) return S4G_OK;
  cudaStream_t s = (cudaStream_t)stream;
  S4G_CUDA(cudaMemsetAsync(grad_in, 0, sizeof(double) * (size_t)B * C * N, s));
  const int MK = M * K;
  dim3 grid((MK + 255) / 256, B);
  s4g::group_backward64_kernel<<<grid, 256, 0, s>>>(grad_out, index, C, N, MK, grad_in);
  S4G_LAUNCH_CHECK("group_points_backward_f64");
  return S4G_OK;
}

extern "C" int s4g_point_search_f64(const double* query, const double* key, int B, int Nq, int Nk, int num_neighbours,
                                    int64_t* index, double* distance, void* stream) {
  S4G_CHECK_ARG(query && key && index && distance, "point_search: null pointer");
  S4G_CHECK_ARG(num_neighbours == 3, "point_search: num_neighbours != 3");
  S4G_CHECK_ARG(Nk >= num_neighbours, "point_search: num_key < num_neighbours");
  S4G_CHECK_ARG(B >= 0 && Nq > 0, "point_search: bad shape");
  S4G_CHECK_ARG(B <= 65535, "point_search: batch too large for one launch");
  if (B == 0) return S4G_OK;
  dim3 grid((Nq + 255) / 256, B);
  s4g::point_search64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(query, key, Nq, Nk, index, distance);
  S4G_LAUNCH_CHECK("point_search_f64");
  return S4G_OK;
}

extern "C" int s4g_interpolate_forward_f64(const double* input, const int64_t* index, const double* weight, int B, int C,
                                           int Nk, int Nq, double* out, void* stream) {
  S4G_CHECK_ARG(input && index && weight && out, "interpolate_forward: null pointer");
  S4G_CHECK_ARG(B >= 0 && C > 0 && Nk > 0 && Nq > 0, "interpolate_forward: bad shape");
  S4G_CHECK_ARG(B <= 65535, "interpolate_forward: batch too large for one launch");
  if (B == 0) return S4G_OK;
  dim3 grid((Nq + 255) / 256, B);
  s4g::interpolate_forward64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(input, index, weight, C, Nk, Nq, out);
  S4G_LAUNCH_CHECK("interpolate_forward_f64");
  return S4G_OK;
}

extern "C" int s4g_interpolate_backward_f64(const double* grad_out, const int64_t* index, const double* weight, int B,
                                            int C, int Nk, int Nq, double* grad_in, void* stream) {
  S4G_CHECK_ARG(grad_out && index && weight && grad_in, "interpolate_backward: null pointer");
  S4G_CHECK_ARG(B >= 0 && C > 0 && Nk > 0 && Nq > 0, "interpolate_backward: bad shape");
  S4G_CHECK_ARG(B <= 65535, "interpolate_backward: batch too large for one launch");
  if (B == 0) return S4G_OK;
  cudaStream_t s = (cudaStream_t)stream;
  S4G_CUDA(cudaMemsetAsync(grad_in, 0, sizeof(double) * (size_t)B * C * Nk, s));
  dim3 grid((Nq + 255) / 256, B);
  s4g::interpolate_backward64_kernel<<<grid, 256, 0, s>>>(grad_out, index, weight, C, Nk, Nq, grad_in);
  S4G_LAUNCH_CHECK("interpolate_backward_f64");
  return S4G_OK;
}
