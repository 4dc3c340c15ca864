// 3-NN search and 3-point interpolation forward/backward in the reference's interface layout.
// Reference: pointnet2_utils/csrc/interpolate_kernel.cu:33-81,92-132 (PointSearch),
// :139-181,191-236 (InterpolateForward), :243-286,296-341 (InterpolateBackward).
//
// point_search: one thread per query; the key cloud is staged once per CTA in shared memory as
// float4 tiles so every key costs one broadcast LDS.128 for 256 queries.  The candidate list is the
// reference's strict-'<' insertion in key order (earlier key wins ties, ascending output).
#include "common.cuh"
#include "grid.cuh"

namespace s4g {

constexpr int kNnThreads = 256;
constexpr int kNnTile = 2048;  // keys per shared-memory tile (32 KB as float4)

__global__ void __launch_bounds__(kNnThreads)
point_search_kernel(const float* __restrict__ query, const float* __restrict__ key, int Nq, int Nk,
                    int64_t* __restrict__ index, float* __restrict__ distance) {
  __shared__ float4 s_key[kNnTile];
  const int b = blockIdx.y;
  const int i = blockIdx.x * kNnThreads + threadIdx.x;
  const bool valid = i < Nq;
  const float* Q = query + (size_t)b * 3 * Nq;
  const float* KX = key + (size_t)b * 3 * Nk;
  const float* KY = KX + Nk;
  const float* KZ = KY + Nk;
  const int iq = valid ? i : Nq - 1;
  const float x1 = Q[iq], y1 = Q[Nq + iq], z1 = Q[2 * Nq + iq];

  // interpolate_kernel.cu:53-54 starts from {1e40 -> +inf, 0, 0} / {-1, 0, 0}: the same state as this all-+inf start
  // once two keys have a finite distance; three_nn_reference_tail restores the reference's slots when fewer do.
  const float inf = __int_as_float(0x7f800000);
  float d0 = inf, d1 = inf, d2 = inf;
  int i0 = -1, i1 = -1, i2 = -1;

  for (int base = 0; base < Nk; base += kNnTile) {
    const int n = min(kNnTile, Nk - base);
    __syncthreads();
    for (int k = threadIdx.x; k < n; k += kNnThreads)
      s_key[k] = make_float4(__ldg(KX + base + k), __ldg(KY + base + k), __ldg(KZ + base + k), 0.f);
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < n; ++k) {
      const float4 p = s_key[k];
      const float d = sqdist(__fsub_rn(x1, p.x), __fsub_rn(y1, p.y), __fsub_rn(z1, p.z));
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
    three_nn_reference_tail(d0, d1, d2, i0, i1, i2, inf);
    int64_t* oi = index + ((size_t)b * Nq + i) * 3;
    float* od = distance + ((size_t)b * Nq + i) * 3;
    oi[0] = i0; oi[1] = i1; oi[2] = i2;
    od[0] = d0; od[1] = d1; od[2] = d2;
  }
}

// out[b,c,n] = fma(in2,w2, fma(in1,w1, fma(in0,w0, 0)))  (interpolate_kernel.cu:167-174)
__global__ void __launch_bounds__(256)
interpolate_forward_kernel(const float* __restrict__ input, const int64_t* __restrict__ index,
                           const float* __restrict__ weight, int C, int Nk, int Nq, float* __restrict__ out) {
  const int b = blockIdx.y;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= Nq) return;
  const int64_t* idx = index + ((size_t)b * Nq + n) * 3;
  const float* w = weight + ((size_t)b * Nq + n) * 3;
  const int64_t j0 = idx[0], j1 = idx[1], j2 = idx[2];
  const float w0 = w[0], w1 = w[1], w2 = w[2];
  const float* in = input + (size_t)b * C * Nk;
  float* o = out + (size_t)b * C * Nq + n;
#pragma unroll 4
  for (int c = 0; c < C; ++c) {
    const float* ic = in + (size_t)c * Nk;
    float v = __fmaf_rn(__ldg(ic + j0), w0, 0.f);
    v = __fmaf_rn(__ldg(ic + j1), w1, v);
    v = __fmaf_rn(__ldg(ic + j2), w2, v);
    o[(size_t)c * Nq] = v;
  }
}

__global__ void __launch_bounds__(256)
interpolate_backward_kernel(const float* __restrict__ grad_out, const int64_t* __restrict__ index,
                            const float* __restrict__ weight, int C, int Nk, int Nq, float* __restrict__ grad_in) {
  const int b = blockIdx.y;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= Nq) return;
  const int64_t* idx = index + ((size_t)b * Nq + n) * 3;
  const float* w = weight + ((size_t)b * Nq + n) * 3;
  const int64_t j0 = idx[0], j1 = idx[1], j2 = idx[2];
  const float w0 = w[0], w1 = w[1], w2 = w[2];
  float* gi = grad_in + (size_t)b * C * Nk;
  const float* go = grad_out + (size_t)b * C * Nq + n;
#pragma unroll 4
  for (int c = 0; c < C; ++c) {
    const float g = __ldg(go + (size_t)c * Nq);
    float* gc = gi + (size_t)c * Nk;
    atomicAdd(gc + j0, __fmul_rn(g, w0));
    atomicAdd(gc + j1, __fmul_rn(g, w1));
    atomicAdd(gc + j2, __fmul_rn(g, w2));
  }
}

}  // namespace s4g

extern "C" int s4g_point_search_f32(const float* query, const float* key, int B, int Nq, int Nk, int num_neighbours,
                                    int64_t* index, float* distance, void* stream) {
  S4G_CHECK_ARG(query && key && index && distance, "point_search: null pointer");
  S4G_CHECK_ARG(num_neighbours == 3, "point_search: num_neighbours != 3");  // interpolate_kernel.cu:105
  S4G_CHECK_ARG(Nk >= num_neighbours, "point_search: num_key < num_neighbours");  // :106
  S4G_CHECK_ARG(B >= 0 && Nq > 0, "point_search: bad shape");
  S4G_CHECK_ARG(B <= 65535, "point_search: batch too large for one launch");
  if (B == 0) return S4G_OK;
  if (Nk >= s4g::kGridKnnMinKeys)
    return s4g::three_nn_grid<0>(query, key, B, Nq, Nk, index, distance, (cudaStream_t)stream);
  dim3 grid((Nq + s4g::kNnThreads - 1) / s4g::kNnThreads, B);
  s4g::point_search_kernel<<<grid, s4g::kNnThreads, 0, (cudaStream_t)stream>>>(query, key, Nq, Nk, index, distance);
  S4G_LAUNCH_CHECK("point_search");
  return S4G_OK;
}

extern "C" int s4g_interpolate_forward_f32(const float* input, const int64_t* index, const float* weight, int B, int C,
                                           int Nk, int Nq, float* out, void* stream) {
  S4G_CHECK_ARG(input && index && weight && out, "interpolate_forward: null pointer");
  S4G_CHECK_ARG(B >= 0 && C > 0 && Nk > 0 && Nq > 0, "interpolate_forward: bad shape");
  S4G_CHECK_ARG(B <= 65535, "interpolate_forward: batch too large for one launch");
  if (B == 0) return S4G_OK;
  dim3 grid((Nq + 255) / 256, B);
  s4g::interpolate_forward_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(input, index, weight, C, Nk, Nq, out);
  S4G_LAUNCH_CHECK("interpolate_forward");
  return S4G_OK;
}

extern "C" int s4g_interpolate_backward_f32(const float* grad_out, const int64_t* index, const float* weight, int B,
                                            int C, int Nk, int Nq, float* grad_in, void* stream) {
  S4G_CHECK_ARG(grad_out && index && weight && grad_in, "interpolate_backward: null pointer");
  S4G_CHECK_ARG(B >= 0 && C > 0 && Nk > 0 && Nq > 0, "interpolate_backward: bad shape");
  S4G_CHECK_ARG(B <= 65535, "interpolate_backward: batch too large for one launch");
  if (B == 0) return S4G_OK;
  cudaStream_t s = (cudaStream_t)stream;
  S4G_CUDA(cudaMemsetAsync(grad_in, 0, sizeof(float) * (size_t)B * C * Nk, s));
  dim3 grid((Nq + 255) / 256, B);
  s4g::interpolate_backward_kernel<<<grid, 256, 0, s>>>(grad_out, index, weight, C, Nk, Nq, grad_in);
  S4G_LAUNCH_CHECK("interpolate_backward");
  return S4G_OK;
}
