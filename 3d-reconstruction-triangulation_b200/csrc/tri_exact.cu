// tri_exact.cu -- kernels whose arithmetic follows the reference's operation order (compiled with
// -fmad=false, see tri_ref.cuh): the trajectory-exact emulation of RayTriangulator's cv::LMSolver
// solve (TRI_RAY_REFERENCE_LM), Triangulator::triangulatePoint over arbitrary camera subsets, and
// Triangulator::getDistFromRay.
#include "tri_batch.cuh"
#include "tri_engine.cuh"
#include "tri_ref.cuh"

namespace tri {

constexpr int EXACT_THREADS = 128;

// ---- RayTriangulator::triangulatePoints, reference LM: one frame per thread ----
template <int PIX>
__global__ void __launch_bounds__(EXACT_THREADS)
ray_reference_kernel(const __grid_constant__ RayRig rig, const char* __restrict__ xy, int64_t row_bytes, int64_t n_frames,
                     int n_use, BatchOut out, unsigned long long* first_bad, int64_t frame_base) {
  const int64_t f = (int64_t)blockIdx.x * EXACT_THREADS + threadIdx.x;
  if (f >= n_frames) return;
  ref::RaySet rs;
  rs.n = 0;
  uint32_t mask = 0;
  for (int c = 0; c < n_use; c++) {
    double x, y; bool ok;
    fetch1<double, PIX>(xy + c * row_bytes, f, x, y, ok);
    if (!ok) continue;
    rs.cam[rs.n] = c;
    ref::make_dir(rig, c, x, y, rs.d[rs.n]);
    rs.n++;
    mask |= 1u << c;
  }
  double X[3] = {0, 0, 0}, err = 0;
  int it = 0;
  if (rs.n >= 2) err = ref::lm_point(rig, rs, X, it);
  else atomicMin(first_bad, (unsigned long long)(frame_base + f));
  if (out.xyz_f32) { float* o = out.xyz_f32 + 3 * f; o[0] = (float)X[0]; o[1] = (float)X[1]; o[2] = (float)X[2]; }
  if (out.xyz_f64) { double* o = out.xyz_f64 + 3 * f; o[0] = X[0]; o[1] = X[1]; o[2] = X[2]; }
  if (out.mask) out.mask[f] = mask;
  if (out.err) out.err[f] = err;
  if (out.iters) out.iters[f] = it;
}

cudaError_t launch_ray_reference(const LaunchCtx& ctx, int pixfmt, const RayRig& rig, const void* d_xy, int n_use,
                                 int64_t n_frames, int64_t cam_stride, const BatchOut& out) {
  if (n_frames <= 0) return cudaSuccess;
  const char* xy = static_cast<const char*>(d_xy);
  const int64_t row_bytes = cam_stride * pix_bytes(pixfmt);
  const unsigned grid = (unsigned)((n_frames + EXACT_THREADS - 1) / EXACT_THREADS);
  switch (pixfmt) {
    case PIX_F32:
      ray_reference_kernel<PIX_F32><<<grid, EXACT_THREADS, 0, ctx.stream>>>(rig, xy, row_bytes, n_frames, n_use, out,
                                                                             ctx.d_first_bad, ctx.frame_base);
      break;
    case PIX_F64:
      ray_reference_kernel<PIX_F64><<<grid, EXACT_THREADS, 0, ctx.stream>>>(rig, xy, row_bytes, n_frames, n_use, out,
                                                                             ctx.d_first_bad, ctx.frame_base);
      break;
    default:
      ray_reference_kernel<PIX_U16><<<grid, EXACT_THREADS, 0, ctx.stream>>>(rig, xy, row_bytes, n_frames, n_use, out,
                                                                             ctx.d_first_bad, ctx.frame_base);
  }
  ++*ctx.launches;
  return cudaGetLastError();
}

// ---- Triangulator::triangulatePoint over arbitrary subsets: one item per thread ----
// solver: 0 = matrix, 1 = ray reference LM, 2 = ray closed form, 3 = ray analytic LM (both via the
// quadratic form, evaluated here in plain double without the folded constants)
__global__ void __launch_bounds__(EXACT_THREADS)
subsets_kernel(const __grid_constant__ DltRig<double> dlt, const __grid_constant__ RayRig rig, int solver, int64_t n_items,
               const int32_t* __restrict__ offs, const int32_t* __restrict__ cam_idx, const double* __restrict__ xy,
               double* __restrict__ xyz, double* __restrict__ err, int32_t* __restrict__ iters, int* bad) {
  const int64_t i = (int64_t)blockIdx.x * EXACT_THREADS + threadIdx.x;
  if (i >= n_items) return;
  const int a = offs[i], n = offs[i + 1] - a;
  double X[3] = {0, 0, 0}, e = 0;
  int it = 0;
  if (n < 1 || n > TRI_MAX_CAMS) {
    atomicExch(bad, 1);
  } else if (solver == 0) {
    int cam[TRI_MAX_CAMS];
    double px[TRI_MAX_CAMS], py[TRI_MAX_CAMS];
    for (int k = 0; k < n; k++) { cam[k] = cam_idx[a + k]; px[k] = xy[2 * (a + k)]; py[k] = xy[2 * (a + k) + 1]; }
    e = ref::dlt_point(dlt, n, cam, px, py, X);
  } else {
    ref::RaySet rs;
    rs.n = n;
    for (int k = 0; k < n; k++) {
      rs.cam[k] = cam_idx[a + k];
      ref::make_dir(rig, rs.cam[k], xy[2 * (a + k)], xy[2 * (a + k) + 1], rs.d[k]);
    }
    if (solver == 1) {
      e = ref::lm_point(rig, rs, X, it);
    } else {
      // closed form: sum (|d|^2 I - d d^T) (p - o) = 0, about the mean origin
      double m[3] = {0, 0, 0};
      for (int k = 0; k < n; k++) for (int j = 0; j < 3; j++) m[j] += rig.pos[rs.cam[k]][j] / n;
      double M[6] = {0, 0, 0, 0, 0, 0}, c[3] = {0, 0, 0};
      for (int k = 0; k < n; k++) {
        const double* d = rs.d[k];
        const double dd = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
        const double o[3] = {rig.pos[rs.cam[k]][0] - m[0], rig.pos[rs.cam[k]][1] - m[1], rig.pos[rs.cam[k]][2] - m[2]};
        const double dot = d[0] * o[0] + d[1] * o[1] + d[2] * o[2];
        M[0] += dd - d[0] * d[0]; M[1] -= d[0] * d[1]; M[2] -= d[0] * d[2];
        M[3] += dd - d[1] * d[1]; M[4] -= d[1] * d[2]; M[5] += dd - d[2] * d[2];
        for (int j = 0; j < 3; j++) c[j] += dd * o[j] - d[j] * dot;
      }
      solve_sym3<double>(M, c, X);
      for (int j = 0; j < 3; j++) X[j] += m[j];
      double S, rmax;
      ref::residual_pass(rig, rs, X, S, rmax, e);
      it = 1;
    }
  }
  xyz[3 * i] = X[0]; xyz[3 * i + 1] = X[1]; xyz[3 * i + 2] = X[2];
  if (err) err[i] = e;
  if (iters) iters[i] = it;
}

__global__ void __launch_bounds__(EXACT_THREADS)
dist_from_ray_kernel(const __grid_constant__ RayRig rig, int64_t n, const int32_t* __restrict__ cam_idx,
                     const double* __restrict__ xy, const double* __restrict__ pts, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * EXACT_THREADS + threadIdx.x;
  if (i >= n) return;
  const double p[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
  out[i] = ref::dist_from_ray(rig, cam_idx[i], xy[2 * i], xy[2 * i + 1], p);
}

}  // namespace tri

using namespace tri;

extern "C" {

int tri_triangulate_subsets(tri_engine* e, int mode, unsigned flags, int64_t n_items, const int32_t* item_offsets,
                            const int32_t* cam_idx, const double* xy, double* xyz, double* err, int32_t* iters) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  if (mode != TRI_MATRIX && mode != TRI_RAY) return fail(TRI_ERR_ARG, "mode must be TRI_MATRIX or TRI_RAY");
  if (n_items < 0) return fail(TRI_ERR_ARG, "negative size");
  if (n_items == 0) return TRI_OK;
  if (!item_offsets || !cam_idx || !xy || !xyz) return fail(TRI_ERR_ARG, "null buffer");
  const int64_t total = item_offsets[n_items];
  for (int64_t i = 0; i < n_items; i++) {
    const int n = item_offsets[i + 1] - item_offsets[i];
    if (n < 2) return fail(TRI_ERR_TOO_FEW, mode == TRI_MATRIX ? "Too few rays are found" : "Too few detections are found");
    if (n > TRI_MAX_CAMS) return fail(TRI_ERR_ARG, "more views in one item than TRI_MAX_CAMS");
  }
  for (int64_t k = 0; k < total; k++)
    if (cam_idx[k] < 0 || cam_idx[k] >= e->n_cams) return fail(TRI_ERR_ARG, "camera index out of range");
  DeviceGuard g(e->device);
  const size_t b_offs = up256(sizeof(int32_t) * (n_items + 1)), b_cam = up256(sizeof(int32_t) * total),
               b_xy = up256(sizeof(double) * 2 * total), b_xyz = up256(sizeof(double) * 3 * n_items),
               b_err = up256(sizeof(double) * n_items), b_it = up256(sizeof(int32_t) * n_items);
  TRI_CUDA(e->scratch.alloc(b_offs + b_cam + b_xy + b_xyz + b_err + b_it + 256));
  char* p = e->scratch.as<char>();
  int32_t* d_offs = (int32_t*)p; p += b_offs;
  int32_t* d_cam = (int32_t*)p; p += b_cam;
  double* d_xy = (double*)p; p += b_xy;
  double* d_xyz = (double*)p; p += b_xyz;
  double* d_err = (double*)p; p += b_err;
  int32_t* d_it = (int32_t*)p; p += b_it;
  int* d_bad = (int*)p;
  cudaStream_t s = e->stream;
  TRI_CUDA(cudaMemcpyAsync(d_offs, item_offsets, sizeof(int32_t) * (n_items + 1), cudaMemcpyHostToDevice, s));
  TRI_CUDA(cudaMemcpyAsync(d_cam, cam_idx, sizeof(int32_t) * total, cudaMemcpyHostToDevice, s));
  TRI_CUDA(cudaMemcpyAsync(d_xy, xy, sizeof(double) * 2 * total, cudaMemcpyHostToDevice, s));
  TRI_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), s));
  const int solver = mode == TRI_MATRIX ? 0 : (flags & TRI_RAY_REFERENCE_LM) ? 1 : 2;
  const unsigned grid = (unsigned)((n_items + EXACT_THREADS - 1) / EXACT_THREADS);
  subsets_kernel<<<grid, EXACT_THREADS, 0, s>>>(e->rig64, e->ray, solver, n_items, d_offs, d_cam, d_xy, d_xyz, d_err, d_it, d_bad);
  e->launches++;
  TRI_CUDA(cudaGetLastError());
  TRI_CUDA(cudaMemcpyAsync(xyz, d_xyz, sizeof(double) * 3 * n_items, cudaMemcpyDeviceToHost, s));
  if (err) TRI_CUDA(cudaMemcpyAsync(err, d_err, sizeof(double) * n_items, cudaMemcpyDeviceToHost, s));
  if (iters) TRI_CUDA(cudaMemcpyAsync(iters, d_it, sizeof(int32_t) * n_items, cudaMemcpyDeviceToHost, s));
  TRI_CUDA(cudaStreamSynchronize(s));
  return TRI_OK;
}

int tri_dist_from_ray(tri_engine* e, int64_t n, const int32_t* cam_idx, const double* xy, const double* points, double* out) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  if (n < 0) return fail(TRI_ERR_ARG, "negative size");
  if (n == 0) return TRI_OK;
  if (!cam_idx || !xy || !points || !out) return fail(TRI_ERR_ARG, "null buffer");
  for (int64_t k = 0; k < n; k++)
    if (cam_idx[k] < 0 || cam_idx[k] >= e->n_cams) return fail(TRI_ERR_ARG, "camera index out of range");
  DeviceGuard g(e->device);
  const size_t b_cam = up256(sizeof(int32_t) * n), b_xy = up256(sizeof(double) * 2 * n), b_p = up256(sizeof(double) * 3 * n),
               b_o = up256(sizeof(double) * n);
  TRI_CUDA(e->scratch.alloc(b_cam + b_xy + b_p + b_o));
  char* p = e->scratch.as<char>();
  int32_t* d_cam = (int32_t*)p; p += b_cam;
  double* d_xy = (double*)p; p += b_xy;
  double* d_p = (double*)p; p += b_p;
  double* d_o = (double*)p;
  cudaStream_t s = e->stream;
  TRI_CUDA(cudaMemcpyAsync(d_cam, cam_idx, sizeof(int32_t) * n, cudaMemcpyHostToDevice, s));
  TRI_CUDA(cudaMemcpyAsync(d_xy, xy, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, s));
  TRI_CUDA(cudaMemcpyAsync(d_p, points, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, s));
  const unsigned grid = (unsigned)((n + EXACT_THREADS - 1) / EXACT_THREADS);
  dist_from_ray_kernel<<<grid, EXACT_THREADS, 0, s>>>(e->ray, n, d_cam, d_xy, d_p, d_o);
  e->launches++;
  TRI_CUDA(cudaGetLastError());
  TRI_CUDA(cudaMemcpyAsync(out, d_o, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  TRI_CUDA(cudaStreamSynchronize(s));
  return TRI_OK;
}

}  // extern "C"
