// Face discriminator helpers of the pose training step (Vid2VidModelD with --add_face_disc, models/vid2vid_model_D.py:148-158,
// 215-230):
//   face_window          : bounding box of the face pixels over all N images -> the clamped fixed-size crop window, in one
//                          launch (per-thread min/max, warp reduction, one atomic per block and value, last-block epilogue)
//   crop_concat_forward  : cat(a[..win], b[..win], dim=1) with the window read from device memory
//   crop_backward        : full-frame gradient of b: the crop's gradient inside the window, zeros outside
#include "v2v_internal.h"

namespace v2v {

namespace {

// win[0..4] = {found, ys, ye, xs, xe}; win[5..9] the accumulators of face_window_kernel, zero between launches:
// max(H - y), max(y + 1), max(W - x), max(x + 1) over the face pixels (0 = none found) and the finished-block count.
constexpr int kAcc = 5;

__device__ __forceinline__ bool face_pixel(const float* __restrict__ p, size_t HW, int predicate) {
  // fp32 comparisons, as torch evaluates `real_A[:, 2] > 0.9` on a float tensor (the literal is rounded to float first)
  if (predicate == 0) return p[2 * HW] > 0.9f;
  const float r = p[0], g = p[HW], b = p[2 * HW];
  return r > 0.19f && r < 0.21f && g < -0.99f && b > -0.61f && b < -0.59f;        // --openpose_only face colour
}

__global__ void __launch_bounds__(256) face_window_kernel(const float* __restrict__ real_A, int N, int C, int H, int W,
                                                          int predicate, int half_y, int half_x, int* __restrict__ win) {
  const size_t HW = (size_t)H * W, total = (size_t)N * HW;
  int a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t n = idx / HW, pix = idx - n * HW;
    if (face_pixel(real_A + n * C * HW + pix, HW, predicate)) {
      const int y = (int)(pix / W), x = (int)(pix - (size_t)y * W);
      a0 = max(a0, H - y);
      a1 = max(a1, y + 1);
      a2 = max(a2, W - x);
      a3 = max(a3, x + 1);
    }
  }
  a0 = __reduce_max_sync(0xffffffffu, a0);
  a1 = __reduce_max_sync(0xffffffffu, a1);
  a2 = __reduce_max_sync(0xffffffffu, a2);
  a3 = __reduce_max_sync(0xffffffffu, a3);
  __shared__ int red[4][8];
  __shared__ bool last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][warp] = a0; red[1][warp] = a1; red[2][warp] = a2; red[3][warp] = a3; }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int nw = blockDim.x >> 5;
    for (int w = 1; w < nw; ++w) {
      a0 = max(a0, red[0][w]); a1 = max(a1, red[1][w]); a2 = max(a2, red[2][w]); a3 = max(a3, red[3][w]);
    }
    if (a1) {                       // a block without face pixels has nothing to add
      atomicMax(win + kAcc + 0, a0);
      atomicMax(win + kAcc + 1, a1);
      atomicMax(win + kAcc + 2, a2);
      atomicMax(win + kAcc + 3, a3);
    }
    __threadfence();
    last = atomicAdd(win + kAcc + 4, 1) == (int)gridDim.x - 1;
  }
  __syncthreads();
  if (!last || threadIdx.x != 0) return;
  __threadfence();
  // last block: read and reset the accumulators, then apply the reference's clamp (vid2vid_model_D.py:221-229)
  const int e0 = atomicExch(win + kAcc + 0, 0), e1 = atomicExch(win + kAcc + 1, 0);
  const int e2 = atomicExch(win + kAcc + 2, 0), e3 = atomicExch(win + kAcc + 3, 0);
  atomicExch(win + kAcc + 4, 0);
  if (!e1) {
    win[0] = win[1] = win[2] = win[3] = win[4] = 0;
    return;
  }
  const int ys = H - e0, ye = e1 - 1, xs = W - e2, xe = e3 - 1;
  int yc = (ys + ye) / 2, xc = (xs + xe) / 2;
  yc = max(half_y, min(H - 1 - half_y, yc));
  xc = max(half_x, min(W - 1 - half_x, xc));
  win[0] = 1;
  win[1] = yc - half_y;
  win[2] = yc + half_y;
  win[3] = xc - half_x;
  win[4] = xc + half_x;
}

// Window origin from device memory, kept inside the frame whatever the buffer holds.
__device__ __forceinline__ void window_origin(const int* __restrict__ win, int H, int W, int Ly, int Lx, int& ys, int& xs) {
  ys = min(max(win[1], 0), H - Ly);
  xs = min(max(win[3], 0), W - Lx);
}

__global__ void __launch_bounds__(256) crop_concat_kernel(const float* __restrict__ a, int Ca, const float* __restrict__ b, int Cb,
                                                          int N, int H, int W, const int* __restrict__ win, int Ly, int Lx,
                                                          float* __restrict__ out) {
  int ys, xs;
  window_origin(win, H, W, Ly, Lx, ys, xs);
  const int Co = Ca + Cb;
  const size_t total = (size_t)N * Co * Ly * Lx;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(idx % Lx);
    size_t r = idx / Lx;
    const int y = (int)(r % Ly);
    r /= Ly;
    const int c = (int)(r % Co);
    const size_t n = r / Co;
    const size_t off = (size_t)(ys + y) * W + xs + x;
    out[idx] = c < Ca ? a[(n * Ca + c) * H * W + off] : b[(n * Cb + (c - Ca)) * H * W + off];
  }
}

__global__ void __launch_bounds__(256) crop_backward_kernel(const float* __restrict__ g, int c_off, int Cb, int N, int H, int W,
                                                            const int* __restrict__ win, int Ly, int Lx, float* __restrict__ gb) {
  int ys, xs;
  window_origin(win, H, W, Ly, Lx, ys, xs);
  const size_t total = (size_t)N * Cb * H * W;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(idx % W);
    size_t r = idx / W;
    const int y = (int)(r % H);
    r /= H;
    const int c = (int)(r % Cb);
    const size_t n = r / Cb;
    const int cy = y - ys, cx = x - xs;
    float v = 0.f;
    if (cy >= 0 && cy < Ly && cx >= 0 && cx < Lx) v = g[((n * (c_off + Cb) + c_off + c) * Ly + cy) * Lx + cx];
    gb[idx] = v;
  }
}

int grid_for(size_t total) {
  size_t b = (total + 255) / 256;
  const size_t cap = 148 * 16;
  return (int)(b < cap ? (b ? b : 1) : cap);
}

}  // namespace

cudaError_t launch_face_window(const float* real_A, int N, int C, int H, int W, int predicate, int half_y, int half_x, int* win,
                               cudaStream_t s) {
  face_window_kernel<<<grid_for((size_t)N * H * W), 256, 0, s>>>(real_A, N, C, H, W, predicate, half_y, half_x, win);
  return cudaGetLastError();
}
cudaError_t launch_crop_concat(const float* a, int Ca, const float* b, int Cb, int N, int H, int W, const int* win, int Ly, int Lx,
                               float* out, cudaStream_t s) {
  crop_concat_kernel<<<grid_for((size_t)N * (Ca + Cb) * Ly * Lx), 256, 0, s>>>(a, Ca, b, Cb, N, H, W, win, Ly, Lx, out);
  return cudaGetLastError();
}
cudaError_t launch_crop_backward(const float* g, int c_off, int Cb, int N, int H, int W, const int* win, int Ly, int Lx, float* gb,
                                 cudaStream_t s) {
  crop_backward_kernel<<<grid_for((size_t)N * Cb * H * W), 256, 0, s>>>(g, c_off, Cb, N, H, W, win, Ly, Lx, gb);
  return cudaGetLastError();
}

}  // namespace v2v
