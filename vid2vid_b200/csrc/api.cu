// extern "C" entry points of the stand-alone operators (group (1) of include/v2v_b200.h).
#include <cmath>
#include <cstring>
#include <string>

#include "../../include/v2v_b200.h"
#include "v2v_internal.h"

namespace v2v {
void set_error(const char* fmt, ...);
cudaError_t launch_correlation(const float*, const float*, float*, int, int, int, int, int, int, int, int, int, cudaStream_t);
cudaError_t launch_resample2d(const float*, const float*, float*, int, int, int, int, int, int, int, cudaStream_t);
cudaError_t launch_channelnorm(const float*, float*, int, int, int, int, int, cudaStream_t);
cudaError_t launch_resample(const float*, const float*, float*, int, int, int, int, int, cudaStream_t);
cudaError_t launch_onehot_edges(const float*, const float*, float*, int, int, int, int, int, cudaStream_t);
cudaError_t launch_avgpool3s2(const float*, float*, int, int, int, cudaStream_t);
cudaError_t launch_flownet_prep(const float*, const float*, long long, long long, float*, float*, float*, int, int, int, float, cudaStream_t);
cudaError_t launch_resize(const float*, float*, float*, int, int, int, int, int, float, float, float, float, float, int, cudaStream_t);
cudaError_t launch_sub_channels(const float*, const float*, float*, int, int, int, int, int, int, cudaStream_t);
cudaError_t launch_flow_conf(const float*, const float*, float*, int, int, int, int, float, cudaStream_t);
cudaError_t launch_ids_window_push(float*, const void*, int, int, int, int, cudaStream_t);
cudaError_t launch_tensor2im_u8(const float*, uint8_t*, int, int, int, cudaStream_t);
cudaError_t launch_l1_fwd(const float*, const float*, const float*, int, int, int, int, double*, float*, cudaStream_t);
cudaError_t launch_l1_bwd(const float*, const float*, const float*, int, int, int, int, const float*, float*, float*, cudaStream_t);
cudaError_t launch_mse_const_fwd(const float*, long long, float, double*, float*, cudaStream_t);
cudaError_t launch_mse_const_bwd(const float*, long long, float, const float*, float*, cudaStream_t);
cudaError_t launch_avgpool3s2_bwd(const float*, float*, int, int, int, cudaStream_t);
cudaError_t launch_resample_bwd(const float*, const float*, const float*, float*, float*, int, int, int, int, int, cudaStream_t);
struct FgLabels { int v[16]; };
cudaError_t launch_fg_mask(const float*, float*, int, int, int, int, int, int, FgLabels, int, cudaStream_t);
cudaError_t launch_face_window(const float*, int, int, int, int, int, int, int, int*, cudaStream_t);
cudaError_t launch_crop_concat(const float*, int, const float*, int, int, int, int, const int*, int, int, float*, cudaStream_t);
cudaError_t launch_crop_backward(const float*, int, int, int, int, int, const int*, int, int, float*, cudaStream_t);
}  // namespace v2v

using namespace v2v;

#define API_CUDA(expr)                                                         \
  do {                                                                         \
    cudaError_t e__ = (expr);                                                  \
    if (e__ != cudaSuccess) {                                                  \
      set_error("%s failed: %s", #expr, cudaGetErrorString(e__));              \
      return (int)e__;                                                         \
    }                                                                          \
  } while (0)
#define API_REQUIRE(cond, ...)     \
  do {                             \
    if (!(cond)) {                 \
      set_error(__VA_ARGS__);      \
      return V2V_ERR_INVALID;      \
    }                              \
  } while (0)

extern "C" {

int v2v_correlation_out_shape(int H, int W, int pad_size, int kernel_size, int max_displacement, int stride1,
                              int stride2, int* outC, int* outH, int* outW) {
  API_REQUIRE(outC && outH && outW && stride1 > 0 && stride2 > 0 && kernel_size > 0, "bad correlation arguments");
  // correlation_cuda.cc:25-38
  const int kernel_radius = (kernel_size - 1) / 2;
  const int border_radius = kernel_radius + max_displacement;
  const int d = (max_displacement / stride2) * 2 + 1;
  *outC = d * d;
  *outH = (int)std::ceil((float)(H + 2 * pad_size - 2 * border_radius) / (float)stride1);
  *outW = (int)std::ceil((float)(W + 2 * pad_size - 2 * border_radius) / (float)stride1);
  return 0;
}

int v2v_correlation_forward(const float* in1, const float* in2, float* out, int N, int C, int H, int W, int pad_size,
                            int kernel_size, int max_displacement, int stride1, int stride2, int corr_type_multiply,
                            v2v_stream_t stream) {
  API_REQUIRE(in1 && in2 && out && N > 0 && C > 0 && H > 0 && W > 0, "null tensor or empty shape");
  API_REQUIRE(kernel_size == 1, "correlation: kernel_size %d unsupported (FlowNetC uses 1)", kernel_size);
  API_REQUIRE(corr_type_multiply == 1, "correlation: only the multiplicative type exists in the reference");
  API_CUDA(launch_correlation(in1, in2, out, N, C, H, W, pad_size, kernel_size, max_displacement, stride1, stride2,
                              reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_resample2d_forward(const float* in1, const float* flow, float* out, int N, int C, int H, int W, int inH,
                           int inW, int kernel_size, v2v_stream_t stream) {
  API_REQUIRE(in1 && flow && out && N > 0 && C > 0 && H > 0 && W > 0, "null tensor or empty shape");
  API_REQUIRE(kernel_size == 1, "resample2d: kernel_size %d unsupported", kernel_size);
  API_CUDA(launch_resample2d(in1, flow, out, N, C, H, W, inH, inW, kernel_size, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_channelnorm_forward(const float* in, float* out, int N, int C, int H, int W, int norm_deg, v2v_stream_t stream) {
  API_REQUIRE(in && out && N > 0 && C > 0 && H > 0 && W > 0, "null tensor or empty shape");
  API_REQUIRE(norm_deg == 2, "channelnorm: norm_deg %d unsupported", norm_deg);
  API_CUDA(launch_channelnorm(in, out, N, C, H, W, norm_deg, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_resample_forward(const float* image, const float* flow, float* out, int N, int C, int H, int W, int align_corners,
                         v2v_stream_t stream) {
  API_REQUIRE(image && flow && out && N > 0 && C > 0 && H > 1 && W > 1, "null tensor or degenerate shape");
  API_CUDA(launch_resample(image, flow, out, N, C, H, W, align_corners, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_onehot_edges(const float* labels, const float* inst, float* out, int F, int label_nc, int use_instance, int H, int W,
                     v2v_stream_t stream) {
  API_REQUIRE(labels && out && F > 0 && label_nc > 0 && H > 0 && W > 0, "null tensor or empty shape");
  API_REQUIRE(!use_instance || inst, "use_instance set but inst is null");
  API_CUDA(launch_onehot_edges(labels, inst, out, F, label_nc, use_instance, H, W, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_avgpool3s2(const float* in, float* out, int P, int H, int W, v2v_stream_t stream) {
  API_REQUIRE(in && out && P > 0 && H > 0 && W > 0, "null tensor or empty shape");
  API_CUDA(launch_avgpool3s2(in, out, P, H, W, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_fg_mask(const float* real_A, float* mask, int B, int T, int C, int H, int W, int t, const int* fg_labels, int n_labels,
                v2v_stream_t stream) {
  API_REQUIRE(real_A && mask && fg_labels && n_labels > 0 && n_labels <= 16, "bad fg_mask arguments");
  API_REQUIRE(t >= 0 && t < T, "frame index out of range");
  FgLabels l{};
  for (int i = 0; i < n_labels; ++i) {
    API_REQUIRE(fg_labels[i] >= 0 && fg_labels[i] < C, "fg label %d out of range for %d channels", fg_labels[i], C);
    l.v[i] = fg_labels[i];
  }
  API_CUDA(launch_fg_mask(real_A, mask, B, T, C, H, W, t, l, n_labels, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_face_window(const float* real_A, int N, int C, int H, int W, int predicate, int half_y, int half_x, int32_t* win,
                    v2v_stream_t stream) {
  API_REQUIRE(real_A && win && N > 0 && C >= 3 && H > 0 && W > 0, "face_window: bad arguments");
  API_REQUIRE(predicate == 0 || predicate == 1, "face_window: predicate %d unknown", predicate);
  API_REQUIRE(half_y >= 0 && half_x >= 0 && 2 * half_y <= H && 2 * half_x <= W,
              "face_window: %dx%d window larger than the %dx%d frame", 2 * half_y, 2 * half_x, H, W);
  API_CUDA(launch_face_window(real_A, N, C, H, W, predicate, half_y, half_x, win, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_crop_concat_forward(const float* a, int Ca, const float* b, int Cb, int N, int H, int W, const int32_t* win, int Ly, int Lx,
                            float* out, v2v_stream_t stream) {
  API_REQUIRE(a && b && win && out && Ca > 0 && Cb > 0 && N > 0, "crop_concat_forward: bad arguments");
  API_REQUIRE(Ly > 0 && Lx > 0 && Ly <= H && Lx <= W, "crop_concat_forward: %dx%d window outside the %dx%d frame", Ly, Lx, H, W);
  API_CUDA(launch_crop_concat(a, Ca, b, Cb, N, H, W, win, Ly, Lx, out, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_crop_backward(const float* grad_out, int c_off, int Cb, int N, int H, int W, const int32_t* win, int Ly, int Lx, float* grad_b,
                      v2v_stream_t stream) {
  API_REQUIRE(grad_out && win && grad_b && c_off >= 0 && Cb > 0 && N > 0, "crop_backward: bad arguments");
  API_REQUIRE(Ly > 0 && Lx > 0 && Ly <= H && Lx <= W, "crop_backward: %dx%d window outside the %dx%d frame", Ly, Lx, H, W);
  API_CUDA(launch_crop_backward(grad_out, c_off, Cb, N, H, W, win, Ly, Lx, grad_b, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_ids_window_push(float* window, const void* frame, int dtype, int T, int H, int W, v2v_stream_t stream) {
  API_REQUIRE(window && frame && dtype >= 0 && dtype <= 2 && T >= 1 && H > 0 && W > 0, "ids_window_push: bad arguments");
  API_CUDA(launch_ids_window_push(window, frame, dtype, T, H, W, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_tensor2im_u8(const float* image, uint8_t* out, int C, int H, int W, v2v_stream_t stream) {
  API_REQUIRE(image && out && C > 0 && H > 0 && W > 0, "tensor2im_u8: bad arguments");
  API_CUDA(launch_tensor2im_u8(image, out, C, H, W, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_flownet_prep(const float* frame0, const float* frame1, int64_t batch_stride, int64_t channel_stride, float* x, float* x1,
                     float* mean_ws, int B, int H, int W, float rgb_max, v2v_stream_t stream) {
  API_REQUIRE(frame0 && frame1 && x && mean_ws && B > 0 && H > 0 && W > 0 && rgb_max != 0.f, "flownet_prep: bad arguments");
  API_CUDA(launch_flownet_prep(frame0, frame1, batch_stride, channel_stride, x, x1, mean_ws, B, H, W, rgb_max,
                               reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_resize(const float* in, float* out, float* out_div, int planes, int h, int w, int H, int W, int mode, int use_scale_factor,
               float mul, float pre_div, float div, v2v_stream_t stream) {
  API_REQUIRE(in && out && planes > 0 && h > 0 && w > 0 && H > 0 && W > 0 && (mode == 0 || mode == 1), "resize: bad arguments");
  API_REQUIRE((!out_div || div != 0.f) && pre_div != 0.f, "resize: division by zero");
  // ATen area_pixel_compute_scale / compute_scales_value: 1 / scale_factor when a scale factor was given, else in / out
  float sh, sw;
  if (use_scale_factor) { sh = 1.0f / ((float)H / (float)h); sw = 1.0f / ((float)W / (float)w); }
  else { sh = (float)h / (float)H; sw = (float)w / (float)W; }
  API_CUDA(launch_resize(in, out, out_div, planes, h, w, H, W, sh, sw, mul, pre_div, div, mode, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_sub_channels(const float* a, const float* b, float* out, int N, int Ca, int c_off, int C, int H, int W, v2v_stream_t stream) {
  API_REQUIRE(a && b && out && N > 0 && C > 0 && c_off >= 0 && c_off + C <= Ca && H > 0 && W > 0, "sub_channels: bad arguments");
  API_CUDA(launch_sub_channels(a, b, out, N, Ca, c_off, C, H, W, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_flow_conf(const float* im1, const float* warped, float* conf, int N, int C, int H, int W, float threshold,
                  v2v_stream_t stream) {
  API_REQUIRE(im1 && warped && conf && N > 0 && C > 0 && H > 0 && W > 0, "flow_conf: bad arguments");
  API_CUDA(launch_flow_conf(im1, warped, conf, N, C, H, W, threshold, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int v2v_l1_loss_forward(const float* a, const float* b, const float* mask, int N, int C, int H, int W, double* sum_ws, float* out,
                        v2v_stream_t stream) {
  API_REQUIRE(a && sum_ws && out && N > 0 && C > 0 && H > 0 && W > 0, "l1_loss: bad arguments");
  API_CUDA(launch_l1_fwd(a, b, mask, N, C, H, W, sum_ws, out, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}
int v2v_l1_loss_backward(const float* a, const float* b, const float* mask, int N, int C, int H, int W, const float* grad_out,
                         float* grad_a, float* grad_b, v2v_stream_t stream) {
  API_REQUIRE(a && grad_out && (grad_a || grad_b), "l1_loss backward: bad arguments");
  API_CUDA(launch_l1_bwd(a, b, mask, N, C, H, W, grad_out, grad_a, grad_b, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}
int v2v_mse_const_forward(const float* x, int64_t numel, float target, double* sum_ws, float* out, v2v_stream_t stream) {
  API_REQUIRE(x && sum_ws && out && numel > 0, "mse_const: bad arguments");
  API_CUDA(launch_mse_const_fwd(x, numel, target, sum_ws, out, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}
int v2v_mse_const_backward(const float* x, int64_t numel, float target, const float* grad_out, float* grad_x, v2v_stream_t stream) {
  API_REQUIRE(x && grad_out && grad_x && numel > 0, "mse_const backward: bad arguments");
  API_CUDA(launch_mse_const_bwd(x, numel, target, grad_out, grad_x, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}
int v2v_avgpool3s2_backward(const float* grad_out, float* grad_in, int P, int H, int W, v2v_stream_t stream) {
  API_REQUIRE(grad_out && grad_in && P > 0 && H > 0 && W > 0, "avgpool3s2 backward: bad arguments");
  API_CUDA(launch_avgpool3s2_bwd(grad_out, grad_in, P, H, W, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}
int v2v_resample_backward(const float* image, const float* flow, const float* grad_out, float* grad_image, float* grad_flow, int N,
                          int C, int H, int W, int align_corners, v2v_stream_t stream) {
  API_REQUIRE(image && flow && grad_out && (grad_image || grad_flow), "resample backward: bad arguments");
  API_CUDA(launch_resample_bwd(image, flow, grad_out, grad_image, grad_flow, N, C, H, W, align_corners,
                               reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

}  // extern "C"
