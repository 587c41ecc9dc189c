// tri_api.cu -- extern "C" layer of libtri_b200.so (include/tri_b200.h): engine life cycle, the
// batch entry points (device-resident and chunked host-buffer pipelines) and the memory helpers.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "tri_engine.cuh"

namespace tri {

static thread_local std::string g_error;
int fail(int status, const std::string& s) {
  g_error = s;
  return status;
}
int cuda_fail(cudaError_t err, const char* what) {
  g_error = std::string(what) + ": " + cudaGetErrorString(err);
  return TRI_ERR_CUDA;
}

// ---- rig constants ---------------------------------------------------------------------------

static bool inv3(const double S[9], double T[9]) {
  double d = S[0] * (S[4] * S[8] - S[5] * S[7]) - S[1] * (S[3] * S[8] - S[5] * S[6]) + S[2] * (S[3] * S[7] - S[4] * S[6]);
  if (!(fabs(d) > 0)) return false;
  d = 1.0 / d;
  T[0] = (S[4] * S[8] - S[5] * S[7]) * d; T[1] = (S[2] * S[7] - S[1] * S[8]) * d; T[2] = (S[1] * S[5] - S[2] * S[4]) * d;
  T[3] = (S[5] * S[6] - S[3] * S[8]) * d; T[4] = (S[0] * S[8] - S[2] * S[6]) * d; T[5] = (S[2] * S[3] - S[0] * S[5]) * d;
  T[6] = (S[3] * S[7] - S[4] * S[6]) * d; T[7] = (S[1] * S[6] - S[0] * S[7]) * d; T[8] = (S[0] * S[4] - S[1] * S[3]) * d;
  return true;
}

// World point closest to all optical axes (axis c: through position_c along the third row of P):
// the FP32 kernels solve in coordinates centred there so that b = x P23 - P03 does not cancel.
static void rig_centre(const tri_engine* e, double c0[3]) {
  double M[9] = {0}, r[3] = {0}, mean[3] = {0};
  for (int c = 0; c < e->n_cams; c++) {
    const double* P = e->cams[c].P;
    double d[3] = {P[8], P[9], P[10]};
    double n = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    if (!(n > 0)) continue;
    for (int k = 0; k < 3; k++) d[k] /= n;
    for (int a = 0; a < 3; a++) {
      double s = 0;
      for (int b = 0; b < 3; b++) {
        double m = (a == b ? 1.0 : 0.0) - d[a] * d[b];
        M[a * 3 + b] += m;
        s += m * e->cams[c].position[b];
      }
      r[a] += s;
    }
    for (int k = 0; k < 3; k++) mean[k] += e->cams[c].position[k] / e->n_cams;
  }
  double Mi[9];
  // guard against (nearly) parallel axes: fall back to the mean camera position
  double tr = M[0] + M[4] + M[8];
  double det = M[0] * (M[4] * M[8] - M[5] * M[7]) - M[1] * (M[3] * M[8] - M[5] * M[6]) + M[2] * (M[3] * M[7] - M[4] * M[6]);
  if (tr > 0 && det > 1e-6 * tr * tr * tr && inv3(M, Mi)) {
    for (int a = 0; a < 3; a++) c0[a] = Mi[a * 3] * r[0] + Mi[a * 3 + 1] * r[1] + Mi[a * 3 + 2] * r[2];
  } else {
    for (int a = 0; a < 3; a++) c0[a] = mean[a];
  }
  for (int a = 0; a < 3; a++)
    if (!isfinite(c0[a])) c0[a] = 0;
}

// Fold one camera's ray model (Triangulator.cpp:15-55) into the affine form of RayFold.
template <typename T>
static void fold_ray(const tri_engine* e, int c, const double c0[3], RayFold<T>& f) {
  const tri_camera& cam = e->cams[c];
  const double w = cam.quat[0], x = cam.quat[1], y = cam.quat[2], z = cam.quat[3];
  // q (0,v) q* for the quaternion as stored (not normalised): |R v| = |q|^2 |v|
  const double R[9] = {w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y),
                       2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                       2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z};
  const double n2 = w * w + x * x + y * y + z * z, n4 = n2 * n2;
  const double W = (double)cam.width, H = (double)cam.height, aspect = W / H;
  const double depth = e->ray.depth[c];
  const double ax = 2 * aspect / W, bx = aspect * (1 / W - 1), ay = 2 / H, by = 1 / H - 1;
  double ob[3], ob2 = 0;
  for (int k = 0; k < 3; k++) {
    f.U0[c][k] = (T)(R[k * 3] * ax);
    f.U1[c][k] = (T)(R[k * 3 + 1] * ay);
    f.U2[c][k] = (T)(R[k * 3] * bx + R[k * 3 + 1] * by + R[k * 3 + 2] * depth);
    ob[k] = cam.position[k] - c0[k];
    ob2 += ob[k] * ob[k];
    f.ob[c][k] = (T)ob[k];
    f.n4ob[c][k] = (T)(n4 * ob[k]);
  }
  f.ax[c] = (T)ax; f.bx[c] = (T)bx; f.ay[c] = (T)ay; f.by[c] = (T)by; f.dd[c] = (T)(depth * depth);
  f.n4[c] = (T)n4;
  f.n4ob2[c] = (T)(n4 * ob2);
}

// RayFold<T>::mask_table (host copy): the presence-only sums of the ray normal equations per 8-bit validity mask,
// accumulated in T in camera order -- exactly what RayPolicy<T>::add_const does view by view.
template <typename T>
static std::vector<T> ray_mask_table(const RayFold<T>& f, int n_cams) {
  std::vector<T> tab((size_t)8 << TRI_RAY_TABLE_CAMS, (T)0);
  const int n = std::min(n_cams, TRI_RAY_TABLE_CAMS);
  for (int m = 0; m < (1 << TRI_RAY_TABLE_CAMS); m++) {
    T cn[3] = {0, 0, 0}, so[3] = {0, 0, 0}, tr = 0, kn = 0;
    for (int c = 0; c < n; c++) {
      if (!(m >> c & 1)) continue;
      for (int k = 0; k < 3; k++) { cn[k] = cn[k] + f.n4ob[c][k]; so[k] = so[k] + f.ob[c][k]; }
      tr = tr + f.n4[c];
      kn = kn + f.n4ob2[c];
    }
    T* row = &tab[(size_t)8 * m];
    row[0] = cn[0]; row[1] = cn[1]; row[2] = cn[2]; row[3] = tr; row[4] = so[0]; row[5] = so[1]; row[6] = so[2]; row[7] = kn;
  }
  return tab;
}
template <typename T>
static cudaError_t upload_ray_table(RayFold<T>& f, int n_cams) {
  const std::vector<T> tab = ray_mask_table(f, n_cams);
  T* d = nullptr;
  cudaError_t err = cudaMalloc((void**)&d, tab.size() * sizeof(T));
  if (err == cudaSuccess) err = cudaMemcpy(d, tab.data(), tab.size() * sizeof(T), cudaMemcpyHostToDevice);
  f.mask_table = d;
  return err;
}

// DltRig<T>::absent (host copy): per group of 8 cameras and per 8-bit set m, what the cameras of m add to the normal
// equations at the canonical pixel (x = y = 0 relative to the rig's pixel origin: rows P[r,0:3], rhs -P[r,3]), accumulated
// in camera order with the kernels' own function (dlt_view of an absent view).
template <typename T>
static std::vector<T> dlt_absent_table(const DltRig<T>& r, int n_cams) {
  const int groups = (n_cams + 7) / 8;
  std::vector<T> tab((size_t)groups * 256 * DLT_TABLE_ROW, (T)0);
  for (int g = 0; g < groups; g++)
    for (int m = 0; m < 256; m++) {
      T M[6] = {0, 0, 0, 0, 0, 0}, v[3] = {0, 0, 0};
      for (int k = 0; k < 8 && 8 * g + k < n_cams; k++)
        if (m >> k & 1) dlt_view<MASK_TABLE>(r.P[8 * g + k], T(0), T(0), false, M, v);
      T* row = &tab[((size_t)g * 256 + m) * DLT_TABLE_ROW];
      for (int k = 0; k < 6; k++) row[k] = M[k];
      for (int k = 0; k < 3; k++) row[6 + k] = v[k];
    }
  return tab;
}
template <typename T>
static cudaError_t upload_dlt_table(DltRig<T>& r, int n_cams) {
  const std::vector<T> tab = dlt_absent_table(r, n_cams);
  T* d = nullptr;
  cudaError_t err = cudaMalloc((void**)&d, tab.size() * sizeof(T));
  if (err == cudaSuccess) err = cudaMemcpy(d, tab.data(), tab.size() * sizeof(T), cudaMemcpyHostToDevice);
  r.absent = d;
  return err;
}

static void build_rigs(tri_engine* e) {
  memset(&e->fold64, 0, sizeof(e->fold64));
  memset(&e->fold32, 0, sizeof(e->fold32));
  memset(&e->rig64, 0, sizeof(e->rig64));
  memset(&e->rig32, 0, sizeof(e->rig32));
  memset(&e->ray, 0, sizeof(e->ray));
  double c0[3];
  rig_centre(e, c0);
  for (int k = 0; k < 3; k++) e->rig32.origin[k] = (float)c0[k];
  // the FP32 origin actually used is the rounded one
  for (int k = 0; k < 3; k++) c0[k] = (double)e->rig32.origin[k];
  for (int c = 0; c < e->n_cams; c++) {
    const tri_camera& cam = e->cams[c];
    for (int k = 0; k < 12; k++) e->rig64.P[c][k] = cam.P[k];
    // FP32 rig: pixel origin at the image centre, world origin at c0 (exact re-parametrisation of
    // the rows of MatrixTriangulator.cpp:16-49, done here in FP64)
    const double px = floor(cam.width / 2.0), py = floor(cam.height / 2.0);
    double Q[12];
    for (int k = 0; k < 4; k++) {
      Q[k] = cam.P[k] - px * cam.P[8 + k];
      Q[4 + k] = cam.P[4 + k] - py * cam.P[8 + k];
      Q[8 + k] = cam.P[8 + k];
    }
    for (int r = 0; r < 3; r++) Q[r * 4 + 3] += Q[r * 4] * c0[0] + Q[r * 4 + 1] * c0[1] + Q[r * 4 + 2] * c0[2];
    for (int k = 0; k < 12; k++) e->rig32.P[c][k] = (float)Q[k];
    e->rig32.pix0[c][0] = (float)px;
    e->rig32.pix0[c][1] = (float)py;
    // ray constants, Triangulator.cpp:27-44
    e->ray.aspect[c] = (double)cam.width / (double)cam.height;
    e->ray.width[c] = (double)cam.width;
    e->ray.height[c] = (double)cam.height;
    e->ray.depth[c] = 1 / tan(cam.fovy_deg * 0.0174533 / 2);
    for (int k = 0; k < 4; k++) e->ray.quat[c][k] = cam.quat[k];
    for (int k = 0; k < 3; k++) e->ray.pos[c][k] = cam.position[k];
    fold_ray(e, c, c0, e->fold64);
    fold_ray(e, c, c0, e->fold32);
  }
  for (int k = 0; k < 3; k++) {
    e->fold64.origin[k] = c0[k];
    e->fold32.origin[k] = (float)c0[k];
  }
}

static int pix_format(unsigned flags, int* fmt) {
  if ((flags & TRI_PIX_F64) && (flags & TRI_PIX_U16)) return fail(TRI_ERR_ARG, "TRI_PIX_F64 and TRI_PIX_U16 are exclusive");
  *fmt = (flags & TRI_PIX_F64) ? PIX_F64 : (flags & TRI_PIX_U16) ? PIX_U16 : PIX_F32;
  return TRI_OK;
}

static int check_batch_args(tri_engine* e, int mode, const void* xy, int n_point_cams, int64_t n_frames,
                            int64_t cam_stride, const tri_batch_out* out, int* n_use) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  if (mode != TRI_MATRIX && mode != TRI_RAY) return fail(TRI_ERR_ARG, "mode must be TRI_MATRIX or TRI_RAY");
  if (n_frames < 0 || n_point_cams < 0) return fail(TRI_ERR_ARG, "negative size");
  if (!out || (n_frames > 0 && !out->xyz_f32 && !out->xyz_f64)) return fail(TRI_ERR_ARG, "no xyz output buffer");
  if (n_frames > 0 && !xy) return fail(TRI_ERR_ARG, "null pixel buffer");
  if (cam_stride < n_frames) return fail(TRI_ERR_DIM, "Every camera should have the same number of points");
  if (mode == TRI_MATRIX) {
    *n_use = std::min(n_point_cams, e->n_cams);  // MatrixTriangulator.cpp:84
  } else {
    if (n_point_cams > e->n_cams)  // RayTriangulator.cpp:65-69 would read past the camera vector
      return fail(TRI_ERR_DIM, "ray mode: more pixel rows than cameras");
    *n_use = n_point_cams;
  }
  return TRI_OK;
}

static int launch_batch(tri_engine* e, const LaunchCtx& ctx, int mode, unsigned flags, int fmt, const void* d_xy, int n_use,
                        int64_t n_frames, int64_t cam_stride, const BatchOut& out) {
  cudaError_t err;
  if (mode == TRI_MATRIX) {
    err = launch_dlt(ctx, (flags & TRI_F32) != 0, fmt, e->rig64, e->rig32, d_xy, n_use, n_frames, cam_stride, out);
  } else {
    if (flags & TRI_RAY_REFERENCE_LM)
      err = launch_ray_reference(ctx, fmt, e->ray, d_xy, n_use, n_frames, cam_stride, out);
    else
      err = launch_ray_fold(ctx, (flags & TRI_RAY_ANALYTIC_LM) != 0, (flags & TRI_F32) != 0, fmt, e->fold64, e->fold32, d_xy,
                            n_use, n_frames, cam_stride, out);
  }
  if (err != cudaSuccess) return cuda_fail(err, "kernel launch");
  return TRI_OK;
}

// A batch without a single pixel row: every frame has too few views -- zero outputs, frame 0 latched.
static int too_few(const LaunchCtx& ctx, int64_t n_frames, const BatchOut& out) {
  TRI_CUDA(cudaMemsetAsync(ctx.d_first_bad, 0, sizeof(unsigned long long), ctx.stream));
  if (out.xyz_f32) TRI_CUDA(cudaMemsetAsync(out.xyz_f32, 0, sizeof(float) * 3 * n_frames, ctx.stream));
  if (out.xyz_f64) TRI_CUDA(cudaMemsetAsync(out.xyz_f64, 0, sizeof(double) * 3 * n_frames, ctx.stream));
  if (out.mask) TRI_CUDA(cudaMemsetAsync(out.mask, 0, sizeof(uint32_t) * n_frames, ctx.stream));
  if (out.err) TRI_CUDA(cudaMemsetAsync(out.err, 0, sizeof(double) * n_frames, ctx.stream));
  if (out.iters) TRI_CUDA(cudaMemsetAsync(out.iters, 0, sizeof(int32_t) * n_frames, ctx.stream));
  return TRI_OK;
}

// Arguments of the robust pair: matrix mode only, its own flag set, a positive threshold, no iteration output.
static int check_robust_args(tri_engine* e, unsigned flags, double max_reproj_px, const void* xy, int n_point_cams, int64_t n_frames,
                             int64_t cam_stride, const tri_batch_out* out, int* n_use) {
  const unsigned allowed = TRI_F32 | TRI_PIX_F64 | TRI_PIX_U16 | TRI_ALLOW_TOO_FEW;
  if (flags & ~allowed) return fail(TRI_ERR_ARG, "robust triangulation accepts TRI_F32, TRI_PIX_F64, TRI_PIX_U16 and TRI_ALLOW_TOO_FEW only");
  if (!(max_reproj_px > 0)) return fail(TRI_ERR_ARG, "max_reproj_px must be > 0");
  if (out && out->iters) return fail(TRI_ERR_ARG, "robust triangulation has no iteration output (iters must be NULL)");
  return check_batch_args(e, TRI_MATRIX, xy, n_point_cams, n_frames, cam_stride, out, n_use);
}

// A host buffer of the staging pipeline: `rows` rows of items of `bytes` bytes, row r starting `r * stride` items after
// `host`.  A null host is an absent buffer: it takes no slot space and is not copied.
struct RowGroup {
  void* host;
  int rows;
  size_t bytes;
  int64_t stride;
};
// A group's rows in a staging slot: row r at d + r * pitch bytes (d is null for an absent group).
struct SlotRows {
  char* d;
  size_t pitch;
};

// Host-buffer pipeline: items stream in chunks through N_SLOTS device staging slots, one CUDA stream each, so the H2D
// copy of a chunk overlaps the kernel of the previous one and the D2H copy of the one before.  For the chunk of n items
// from f0, on its slot's stream: the [f0, f0 + n) slice of every input row goes H2D, `launch(ctx, n, in, out)` runs on
// the slot's rows, and the slice of every output row comes back D2H, each in the order the groups are listed.
template <class Launch>
static int run_staged(tri_engine* e, int64_t n_items, int64_t chunk, const std::vector<RowGroup>& in,
                      const std::vector<RowGroup>& out, Launch launch) {
  const int n_slots = n_items > chunk ? N_SLOTS : 1;
  // slot buffers: the present groups back to back, every row at a 256-byte aligned offset
  auto pitch = [&](const RowGroup& g) { return up256((size_t)chunk * g.bytes); };
  auto bytes = [&](const std::vector<RowGroup>& groups) {
    size_t b = 0;
    for (const RowGroup& g : groups) b += g.host ? g.rows * pitch(g) : 0;
    return b;
  };
  auto place = [&](const std::vector<RowGroup>& groups, DevBuf& buf) {
    std::vector<SlotRows> rows;
    char* p = buf.as<char>();
    for (const RowGroup& g : groups) {
      rows.push_back({g.host ? p : nullptr, pitch(g)});
      if (g.host) p += g.rows * pitch(g);
    }
    return rows;
  };
  auto copy = [&](const std::vector<RowGroup>& groups, const std::vector<SlotRows>& rows, int64_t f0, int64_t n, bool h2d,
                  cudaStream_t stream) -> int {
    for (size_t i = 0; i < groups.size(); i++)
      for (int r = 0; rows[i].d && r < groups[i].rows; r++) {
        char* h = static_cast<char*>(groups[i].host) + (r * groups[i].stride + f0) * groups[i].bytes;
        char* d = rows[i].d + r * rows[i].pitch;
        TRI_CUDA(cudaMemcpyAsync(h2d ? d : h, h2d ? h : d, (size_t)n * groups[i].bytes,
                                 h2d ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost, stream));
      }
    return TRI_OK;
  };
  // the chunk loop; on any failure the copies already queued into the caller's buffers are drained before returning
  auto run = [&]() -> int {
    for (int i = 0; i < n_slots; i++) {
      TRI_CUDA(e->slots[i].in.alloc(bytes(in)));
      TRI_CUDA(e->slots[i].out.alloc(bytes(out)));
    }
    int k = 0, st;
    for (int64_t f0 = 0; f0 < n_items; f0 += chunk, k++) {
      Slot& s = e->slots[k % n_slots];
      const int64_t n = std::min(chunk, n_items - f0);
      const std::vector<SlotRows> d_in = place(in, s.in), d_out = place(out, s.out);
      TRI_CUDA(cudaStreamSynchronize(s.stream));  // slot free (its previous D2H has landed)
      if ((st = copy(in, d_in, f0, n, true, s.stream)) != TRI_OK) return st;
      if ((st = launch(e->ctx(s.stream, f0, true), n, d_in.data(), d_out.data())) != TRI_OK) return st;
      if ((st = copy(out, d_out, f0, n, false, s.stream)) != TRI_OK) return st;
    }
    for (int i = 0; i < n_slots; i++) TRI_CUDA(cudaStreamSynchronize(e->slots[i].stream));
    return TRI_OK;
  };
  const int st = run();
  if (st != TRI_OK) {
    const std::string why = g_error;
    for (int i = 0; i < n_slots; i++) cudaStreamSynchronize(e->slots[i].stream);  // nothing is left in flight into the caller's memory
    cudaGetLastError();
    return fail(st, why);
  }
  return TRI_OK;
}

// Host-buffer batch (plain or robust): the pixel rows in, the outputs asked for back, through the staging pipeline.
// `launch(ctx, d_xy, n, cam_stride, out)` solves one chunk already on the device.
template <class Launch>
static int run_batch_host(tri_engine* e, unsigned flags, int fmt, const void* xy, int n_use, int64_t n_frames, int64_t cam_stride,
                          int64_t chunk, const tri_batch_out* out, int64_t* first_bad_frame, const char* too_few_msg, Launch launch) {
  const size_t pb = pix_bytes(fmt);
  if (n_frames <= chunk) chunk = (n_frames + 1) / 2 * 2;  // one chunk
  unsigned long long* latch = e->d_first_bad + 1;  // the host path's own latch: a pending one of the device entry point stays
  TRI_CUDA(cudaMemsetAsync(latch, 0xff, sizeof(unsigned long long), e->slots[0].stream));
  TRI_CUDA(cudaStreamSynchronize(e->slots[0].stream));
  const int st = run_staged(
      e, n_frames, chunk, {{const_cast<void*>(xy), n_use, pb, cam_stride}},
      {{out->xyz_f32, 1, 12, 0}, {out->xyz_f64, 1, 24, 0}, {out->mask, 1, 4, 0}, {out->err, 1, 8, 0}, {out->iters, 1, 4, 0}},
      [&](const LaunchCtx& ctx, int64_t n, const SlotRows* d_in, const SlotRows* d_out) {
        const BatchOut o{(float*)d_out[0].d, (double*)d_out[1].d, (uint32_t*)d_out[2].d, (double*)d_out[3].d, (int32_t*)d_out[4].d};
        if (n_use == 0) return too_few(ctx, n, o);
        return launch(ctx, (const void*)d_in[0].d, n, (int64_t)(d_in[0].pitch / pb), o);
      });
  if (st != TRI_OK) {
    cudaMemset(latch, 0xff, sizeof(unsigned long long));
    cudaGetLastError();
    return st;
  }
  unsigned long long v = 0;
  TRI_CUDA(cudaMemcpy(&v, latch, sizeof(v), cudaMemcpyDeviceToHost));
  if (v != ~0ull) {
    TRI_CUDA(cudaMemset(latch, 0xff, sizeof(v)));
    if (first_bad_frame) *first_bad_frame = (int64_t)v;
    if (!(flags & TRI_ALLOW_TOO_FEW)) return fail(TRI_ERR_TOO_FEW, too_few_msg);
  }
  return TRI_OK;
}

// Arguments of the projection pair (tri_project_points*).
static int check_project_args(tri_engine* e, unsigned flags, const float* xyz_f32, const double* xyz_f64, int64_t n_points,
                              const void* xy, int64_t cam_stride, const uint32_t* mask, int* fmt) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  if (flags & ~(unsigned)(TRI_F32 | TRI_PIX_F64 | TRI_PIX_U16))
    return fail(TRI_ERR_ARG, "projection accepts TRI_F32, TRI_PIX_F64 and TRI_PIX_U16 only");
  int st = pix_format(flags, fmt);
  if (st != TRI_OK) return st;
  if (n_points < 0) return fail(TRI_ERR_ARG, "negative size");
  if (n_points > 0 && (!xyz_f32) == (!xyz_f64)) return fail(TRI_ERR_ARG, "exactly one of xyz_f32 / xyz_f64 must be given");
  if (n_points > 0 && !xy && !mask) return fail(TRI_ERR_ARG, "no output buffer (xy and mask are both null)");
  if (cam_stride < n_points) return fail(TRI_ERR_DIM, "Every camera should have the same number of points");
  if (*fmt == PIX_U16)
    for (int c = 0; c < e->n_cams; c++)
      if (e->cams[c].width > 65535 || e->cams[c].height > 65535)
        return fail(TRI_ERR_ARG, "TRI_PIX_U16: a camera is larger than 65535 pixels, its pixels could collide with the missing marker");
  return TRI_OK;
}

}  // namespace tri

using namespace tri;

extern "C" {

int tri_version(void) { return 100; }
const char* tri_last_error(void) { return g_error.c_str(); }

int tri_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int tri_create(int n_cams, const tri_camera* cams, int device, tri_engine** out) {
  if (!out) return fail(TRI_ERR_ARG, "null out pointer");
  *out = nullptr;
  if (n_cams < 1 || n_cams > TRI_MAX_CAMS || !cams) return fail(TRI_ERR_ARG, "n_cams must be in [1, TRI_MAX_CAMS]");
  int n_dev = tri_device_count();
  if (n_dev <= 0) return fail(TRI_ERR_NO_DEVICE, "no CUDA device: the engine has no CPU path");
  if (device < 0 || device >= n_dev) return fail(TRI_ERR_ARG, "device index out of range");
  for (int c = 0; c < n_cams; c++)
    if (cams[c].width <= 0 || cams[c].height <= 0) return fail(TRI_ERR_ARG, "camera width/height must be positive");
  DeviceGuard g(device);
  cudaDeviceProp prop;
  TRI_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(TRI_ERR_NO_DEVICE, "libtri_b200 is built for sm_100a (B200) only");
  tri_engine* e = new tri_engine();
  e->device = device;
  e->n_cams = n_cams;
  e->sm_count = prop.multiProcessorCount;
  memcpy(e->cams, cams, sizeof(tri_camera) * n_cams);
  build_rigs(e);
  cudaError_t err = cudaMalloc((void**)&e->d_first_bad, 2 * sizeof(unsigned long long));
  if (err == cudaSuccess) err = cudaMemset(e->d_first_bad, 0xff, 2 * sizeof(unsigned long long));
  if (err == cudaSuccess) err = upload_dlt_table(e->rig32, n_cams);
  if (err == cudaSuccess) err = upload_ray_table(e->fold64, n_cams);
  if (err == cudaSuccess) err = upload_ray_table(e->fold32, n_cams);
  if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
  for (int i = 0; i < N_SLOTS && err == cudaSuccess; i++) err = cudaStreamCreateWithFlags(&e->slots[i].stream, cudaStreamNonBlocking);
  if (err != cudaSuccess) {
    int st = cuda_fail(err, "tri_create");
    tri_destroy(e);
    return st;
  }
  *out = e;
  return TRI_OK;
}

void tri_destroy(tri_engine* e) {
  if (!e) return;
  DeviceGuard g(e->device);
  cudaDeviceSynchronize();
  for (int i = 0; i < N_SLOTS; i++)
    if (e->slots[i].stream) cudaStreamDestroy(e->slots[i].stream);
  if (e->cls_work && e->cls_work_free) e->cls_work_free(e->cls_work);
  if (e->stream) cudaStreamDestroy(e->stream);
  if (e->d_first_bad) cudaFree(e->d_first_bad);
  if (e->rig32.absent) cudaFree(const_cast<float*>(e->rig32.absent));
  if (e->fold64.mask_table) cudaFree(const_cast<double*>(e->fold64.mask_table));
  if (e->fold32.mask_table) cudaFree(const_cast<float*>(e->fold32.mask_table));
  delete e;  // the DevBuf members free the staging slots and the scratch
}

int tri_engine_device(const tri_engine* e) { return e ? e->device : -1; }
int tri_engine_cameras(const tri_engine* e) { return e ? e->n_cams : 0; }
int64_t tri_kernel_launches(const tri_engine* e) { return e ? e->launches : 0; }

int tri_triangulate_points_device(tri_engine* e, int mode, unsigned flags, const void* d_xy, int n_point_cams,
                                  int64_t n_frames, int64_t cam_stride, const tri_batch_out* d_out, void* stream) {
  int n_use = 0, fmt = 0;
  int st = check_batch_args(e, mode, d_xy, n_point_cams, n_frames, cam_stride, d_out, &n_use);
  if (st != TRI_OK) return st;
  if ((st = pix_format(flags, &fmt)) != TRI_OK) return st;
  if (n_frames == 0) return TRI_OK;
  DeviceGuard g(e->device);
  BatchOut out{d_out->xyz_f32, d_out->xyz_f64, d_out->mask, d_out->err, d_out->iters};
  if (n_use == 0) return too_few(e->ctx((cudaStream_t)stream), n_frames, out);
  return launch_batch(e, e->ctx((cudaStream_t)stream), mode, flags, fmt, d_xy, n_use, n_frames, cam_stride, out);
}

int tri_enable_peer_access(tri_engine* e, int peer_device) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  if (peer_device == e->device) return TRI_OK;
  DeviceGuard g(e->device);
  int can = 0;
  TRI_CUDA(cudaDeviceCanAccessPeer(&can, e->device, peer_device));
  if (!can) return fail(TRI_ERR_ARG, "no peer access between these GPUs");
  cudaError_t err = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (err == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return TRI_OK; }
  if (err != cudaSuccess) return cuda_fail(err, "cudaDeviceEnablePeerAccess");
  return TRI_OK;
}

int tri_ipc_export(tri_engine* e, void* d_ptr, unsigned char handle[64]) {
  if (!e || !d_ptr || !handle) return fail(TRI_ERR_ARG, "null pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  DeviceGuard g(e->device);
  cudaIpcMemHandle_t h;
  TRI_CUDA(cudaIpcGetMemHandle(&h, d_ptr));
  memcpy(handle, &h, 64);
  return TRI_OK;
}

int tri_ipc_open(tri_engine* e, const unsigned char handle[64], void** d_ptr) {
  if (!e || !d_ptr || !handle) return fail(TRI_ERR_ARG, "null pointer");
  DeviceGuard g(e->device);
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  TRI_CUDA(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return TRI_OK;
}

int tri_ipc_close(tri_engine* e, void* d_ptr) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  DeviceGuard g(e->device);
  if (d_ptr) TRI_CUDA(cudaIpcCloseMemHandle(d_ptr));
  return TRI_OK;
}

int tri_copy_device(tri_engine* e, void* d_dst, const void* d_src, uint64_t bytes) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  DeviceGuard g(e->device);
  TRI_CUDA(cudaMemcpy(d_dst, d_src, bytes, cudaMemcpyDefault));
  return TRI_OK;
}

int tri_device_status(tri_engine* e, void* stream, int64_t* first_bad_frame) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  DeviceGuard g(e->device);
  unsigned long long v = 0;
  TRI_CUDA(cudaMemcpyAsync(&v, e->d_first_bad, sizeof(v), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  TRI_CUDA(cudaMemsetAsync(e->d_first_bad, 0xff, sizeof(v), (cudaStream_t)stream));
  TRI_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  if (v != ~0ull) {
    if (first_bad_frame) *first_bad_frame = (int64_t)v;
    return fail(TRI_ERR_TOO_FEW, "a frame has fewer than 2 detections");
  }
  if (first_bad_frame) *first_bad_frame = -1;
  return TRI_OK;
}

int tri_triangulate_points(tri_engine* e, int mode, unsigned flags, const void* xy, int n_point_cams, int64_t n_frames,
                           int64_t cam_stride, const tri_batch_out* out, int64_t* first_bad_frame) {
  int n_use = 0, fmt = 0;
  int st = check_batch_args(e, mode, xy, n_point_cams, n_frames, cam_stride, out, &n_use);
  if (st != TRI_OK) return st;
  if ((st = pix_format(flags, &fmt)) != TRI_OK) return st;
  if (first_bad_frame) *first_bad_frame = -1;
  if (n_frames == 0) return TRI_OK;
  DeviceGuard g(e->device);
  // chunk: large enough to run the copy engines at full rate, small enough to pipeline
  int64_t chunk = n_frames >= (16 << 20) ? (4 << 20) : (1 << 20);  // measured: 4 Mi-frame chunks run PCIe at 63 GB/s, 1 Mi at 60.6
  if (mode == TRI_RAY && (flags & TRI_RAY_REFERENCE_LM)) chunk = 1 << 18;
  return run_batch_host(e, flags, fmt, xy, n_use, n_frames, cam_stride, chunk, out, first_bad_frame,
                        mode == TRI_MATRIX ? "Too few rays are found" : "Too few detections are found",
                        [&](const LaunchCtx& ctx, const void* d_in, int64_t n, int64_t stride, const BatchOut& o) {
                          return launch_batch(e, ctx, mode, flags, fmt, d_in, n_use, n, stride, o);
                        });
}

int tri_triangulate_points_robust_device(tri_engine* e, unsigned flags, double max_reproj_px, const void* d_xy, int n_point_cams,
                                         int64_t n_frames, int64_t cam_stride, const tri_batch_out* d_out, void* stream) {
  int n_use = 0, fmt = 0;
  int st = check_robust_args(e, flags, max_reproj_px, d_xy, n_point_cams, n_frames, cam_stride, d_out, &n_use);
  if (st != TRI_OK) return st;
  if ((st = pix_format(flags, &fmt)) != TRI_OK) return st;
  if (n_frames == 0) return TRI_OK;
  DeviceGuard g(e->device);
  BatchOut out{d_out->xyz_f32, d_out->xyz_f64, d_out->mask, d_out->err, nullptr};
  if (n_use == 0) return too_few(e->ctx((cudaStream_t)stream), n_frames, out);
  const cudaError_t err = launch_robust(e->ctx((cudaStream_t)stream), (flags & TRI_F32) != 0, fmt, e->rig64, e->rig32, max_reproj_px,
                                        d_xy, n_use, n_frames, cam_stride, out);
  return err == cudaSuccess ? TRI_OK : cuda_fail(err, "kernel launch");
}

int tri_triangulate_points_robust(tri_engine* e, unsigned flags, double max_reproj_px, const void* xy, int n_point_cams,
                                  int64_t n_frames, int64_t cam_stride, const tri_batch_out* out, int64_t* first_bad_frame) {
  int n_use = 0, fmt = 0;
  int st = check_robust_args(e, flags, max_reproj_px, xy, n_point_cams, n_frames, cam_stride, out, &n_use);
  if (st != TRI_OK) return st;
  if ((st = pix_format(flags, &fmt)) != TRI_OK) return st;
  if (first_bad_frame) *first_bad_frame = -1;
  if (n_frames == 0) return TRI_OK;
  DeviceGuard g(e->device);
  // the solve is compute-bound (pairs x views per frame), so the copies hide under it at the plain path's 1 Mi-frame chunk
  return run_batch_host(e, flags, fmt, xy, n_use, n_frames, cam_stride, (int64_t)1 << 20, out, first_bad_frame,
                        "Too few rays are found",
                        [&](const LaunchCtx& ctx, const void* d_in, int64_t n, int64_t stride, const BatchOut& o) {
                          const cudaError_t err = launch_robust(ctx, (flags & TRI_F32) != 0, fmt, e->rig64, e->rig32, max_reproj_px,
                                                                d_in, n_use, n, stride, o);
                          return err == cudaSuccess ? TRI_OK : cuda_fail(err, "kernel launch");
                        });
}

int tri_project_points_device(tri_engine* e, unsigned flags, const float* d_xyz_f32, const double* d_xyz_f64, int64_t n_points,
                              void* d_xy, int64_t cam_stride, uint32_t* d_mask, void* stream) {
  int fmt = 0;
  const int st = check_project_args(e, flags, d_xyz_f32, d_xyz_f64, n_points, d_xy, cam_stride, d_mask, &fmt);
  if (st != TRI_OK || n_points == 0) return st;
  DeviceGuard g(e->device);
  const cudaError_t err = launch_project(e->ctx((cudaStream_t)stream), (flags & TRI_F32) != 0, fmt, e->rig64, e->rig32, e->cams, e->n_cams,
                                         d_xyz_f32, d_xyz_f64, n_points, d_xy, cam_stride, d_mask);
  return err == cudaSuccess ? TRI_OK : cuda_fail(err, "kernel launch");
}

int tri_project_points(tri_engine* e, unsigned flags, const float* xyz_f32, const double* xyz_f64, int64_t n_points, void* xy,
                       int64_t cam_stride, uint32_t* mask) {
  int fmt = 0;
  const int st = check_project_args(e, flags, xyz_f32, xyz_f64, n_points, xy, cam_stride, mask, &fmt);
  if (st != TRI_OK || n_points == 0) return st;
  DeviceGuard g(e->device);
  const size_t pb = pix_bytes(fmt), in_pp = xyz_f32 ? 12 : 24;
  const int nc = e->n_cams;
  // ~64 MB of output rows per slot: large enough for full-rate copies, small enough to pipeline
  const size_t out_pp = (xy ? nc * pb : 0) + (mask ? 4 : 0);
  int64_t chunk = std::min<int64_t>(std::max<int64_t>((int64_t)((64u << 20) / out_pp) / 256 * 256, 1 << 16), 4 << 20);
  if (n_points <= chunk) chunk = n_points;
  const void* xyz = xyz_f32 ? (const void*)xyz_f32 : (const void*)xyz_f64;
  return run_staged(e, n_points, chunk, {{const_cast<void*>(xyz), 1, in_pp, 0}}, {{xy, nc, pb, cam_stride}, {mask, 1, 4, 0}},
                    [&](const LaunchCtx& ctx, int64_t n, const SlotRows* d_in, const SlotRows* d_out) {
                      const cudaError_t err = launch_project(ctx, (flags & TRI_F32) != 0, fmt, e->rig64, e->rig32, e->cams, nc,
                                                             xyz_f32 ? (const float*)d_in[0].d : nullptr,
                                                             xyz_f64 ? (const double*)d_in[0].d : nullptr, n, d_out[0].d,
                                                             (int64_t)(d_out[0].pitch / pb), (uint32_t*)d_out[1].d);
                      return err == cudaSuccess ? TRI_OK : cuda_fail(err, "kernel launch");
                    });
}

int tri_triangulate_points_multi(tri_engine* const* engines, int n_engines, int mode, unsigned flags, const void* xy,
                                 int n_point_cams, int64_t n_frames, int64_t cam_stride, const tri_batch_out* out,
                                 int64_t* first_bad_frame) {
  if (!engines || n_engines < 1) return fail(TRI_ERR_ARG, "no engines");
  for (int g = 0; g < n_engines; g++)
    if (!engines[g] || engines[g]->n_cams != engines[0]->n_cams) return fail(TRI_ERR_ARG, "engines must hold the same rig");
  if (n_engines == 1) return tri_triangulate_points(engines[0], mode, flags, xy, n_point_cams, n_frames, cam_stride, out, first_bad_frame);
  int fmt = 0, n_use = 0;
  int st = check_batch_args(engines[0], mode, xy, n_point_cams, n_frames, cam_stride, out, &n_use);
  if (st != TRI_OK) return st;
  if ((st = pix_format(flags, &fmt)) != TRI_OK) return st;
  const size_t pb = pix_bytes(fmt);
  std::vector<int64_t> bad(n_engines, -1);
  auto cut = [&](int g) {  // even boundaries keep every shard's rows vector-aligned
    int64_t b = n_frames * g / n_engines;
    return g >= n_engines ? n_frames : std::min<int64_t>(n_frames, b + (b & 1));
  };
  st = fan_out(n_engines, [&](int g) -> int {
    const int64_t b = cut(g), e = cut(g + 1);
    if (e <= b) return TRI_OK;
    tri_batch_out o{out->xyz_f32 ? out->xyz_f32 + 3 * b : nullptr, out->xyz_f64 ? out->xyz_f64 + 3 * b : nullptr,
                    out->mask ? out->mask + b : nullptr, out->err ? out->err + b : nullptr, out->iters ? out->iters + b : nullptr};
    const int rc = tri_triangulate_points(engines[g], mode, flags | TRI_ALLOW_TOO_FEW, static_cast<const char*>(xy) + (size_t)b * pb,
                                          n_point_cams, e - b, cam_stride, &o, &bad[g]);
    if (bad[g] >= 0) bad[g] += b;
    return rc;
  });
  if (st != TRI_OK) return st;
  int64_t first = -1;
  for (int g = 0; g < n_engines; g++)
    if (bad[g] >= 0 && (first < 0 || bad[g] < first)) first = bad[g];
  if (first_bad_frame) *first_bad_frame = first;
  if (first >= 0 && !(flags & TRI_ALLOW_TOO_FEW))
    return fail(TRI_ERR_TOO_FEW, mode == TRI_MATRIX ? "Too few rays are found" : "Too few detections are found");
  return TRI_OK;
}

// ---- memory helpers ----------------------------------------------------------------------------

int tri_host_alloc(void** p, uint64_t bytes) {
  if (!p) return fail(TRI_ERR_ARG, "null pointer");
  TRI_CUDA(cudaHostAlloc(p, bytes ? bytes : 1, cudaHostAllocPortable));
  return TRI_OK;
}
int tri_host_free(void* p) {
  if (p) TRI_CUDA(cudaFreeHost(p));
  return TRI_OK;
}
int tri_device_alloc(tri_engine* e, void** p, uint64_t bytes) {
  if (!e || !p) return fail(TRI_ERR_ARG, "null pointer");
  DeviceGuard g(e->device);
  TRI_CUDA(cudaMalloc(p, bytes ? bytes : 1));
  return TRI_OK;
}
int tri_device_free(tri_engine* e, void* p) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  DeviceGuard g(e->device);
  if (p) TRI_CUDA(cudaFree(p));
  return TRI_OK;
}
int tri_copy_to_device(tri_engine* e, void* d_dst, const void* h_src, uint64_t bytes) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  DeviceGuard g(e->device);
  TRI_CUDA(cudaMemcpy(d_dst, h_src, bytes, cudaMemcpyHostToDevice));
  return TRI_OK;
}
int tri_copy_to_host(tri_engine* e, void* h_dst, const void* d_src, uint64_t bytes) {
  if (!e) return fail(TRI_ERR_ARG, "null engine");
  DeviceGuard g(e->device);
  TRI_CUDA(cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost));
  return TRI_OK;
}

}  // extern "C"
