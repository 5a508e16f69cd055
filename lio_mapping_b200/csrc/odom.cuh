// Device pieces of Estimator::CalculateLaserOdom (src/imu_processor/Estimator.cc:1242-1359) and of the scan-to-map loops
// built on it (PointMapping.cc:609-715, MapBuilder.cc:873-1011), shared by the stand-alone reduce / solve kernels
// (estimator.cu) and by the fused tail of the k-NN kernel (knn.cu).  Compile the including unit with -fmad=false.
#pragma once
#include "knn.cuh"
#include "qr.cuh"

namespace lio {

struct OdomState {
  double AtA[36];
  double AtB[6];
  float matP[36];
  int degenerate;
  int done;
  int iter;
  unsigned counter;
};

// Workspace + driver of the scan-to-map optimisation on device-resident clouds (estimator.cu); shared by the host-array
// parity entry lio_scan_to_map_host and by the cube-map context (cubemap.cu).
struct ScanToMapWork {
  CellHash hc, hs;
  KnnWork w;
  FeatureOut fo;
  int *d_n = nullptr;          // [0] Kc [1] Ks [4] feature count
  TransformF *d_tf = nullptr;
  OdomState *d_odom = nullptr;
  double *d_partial = nullptr;
  float *d_z = nullptr;
  unsigned char *h_stage = nullptr;   // pinned: the counts, point_on_z_axis_ and the start pose uploaded by scan_to_map_run
  int cap_feat = 0;
  int init(int cap_corner_map, int cap_surf_map, int cap_queries);
  void destroy();
};
int scan_to_map_run(ScanToMapWork &W, const float4 *d_cmap, int Kc, const float4 *d_smap, int Ks, const float4 *d_corner, const int *d_nc,
                    int Mc_max, const float4 *d_surf, const int *d_ns, int Ms_max, float *tf7, float min_match_sq_dis, float min_plane_dis,
                    int max_iter, double delta_r_abort, double delta_t_abort, int variant, int *n_out, int *iters, int sm, cudaStream_t st,
                    CallStats *stats = nullptr);

// rot.toRotationMatrix() of the (possibly un-normalised) float quaternion
__device__ __forceinline__ void odom_rotation(const TransformF &tf, float (&R)[9]) {
  const float tx = 2.f * tf.qx, ty = 2.f * tf.qy, tz = 2.f * tf.qz;
  const float twx = tx * tf.qw, twy = ty * tf.qw, twz = tz * tf.qw, txx = tx * tf.qx, txy = ty * tf.qx, txz = tz * tf.qx;
  const float tyy = ty * tf.qy, tyz = tz * tf.qy, tzz = tz * tf.qz;
  R[0] = 1.f - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
  R[3] = txy + twz; R[4] = 1.f - (txx + tzz); R[5] = tyz - twx;
  R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1.f - (txx + tyy);
}

__device__ __forceinline__ void odom_qmul_vec(float qx, float qy, float qz, float qw, float vx, float vy, float vz, float &ox, float &oy, float &oz) {
  float ux = qy * vz - qz * vy, uy = qz * vx - qx * vz, uz = qx * vy - qy * vx;
  ux += ux; uy += uy; uz += uz;
  float cx = qy * uz - qz * uy, cy = qz * ux - qx * uz, cz = qx * uy - qy * ux;
  ox = vx + ux * qw + cx; oy = vy + uy * qw + cy; oz = vz + uz * qw + cz;
}

// One feature of CalculateLaserOdom (mode 0): Jacobian row J = [-w^T R [p]x | w^T] and d2 = w . (R p + t) + b
// (Estimator.cc:1282-1300), float arithmetic in the reference's order.
__device__ __forceinline__ void odom_row(const TransformF &tf, const float (&R)[9], float4 p, float4 c, float (&row)[6], float &d2) {
  float RS[9];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    RS[r * 3 + 0] = R[r * 3 + 1] * p.z + R[r * 3 + 2] * (-p.y);
    RS[r * 3 + 1] = R[r * 3 + 0] * (-p.z) + R[r * 3 + 2] * p.x;
    RS[r * 3 + 2] = R[r * 3 + 0] * p.y + R[r * 3 + 1] * (-p.x);
  }
#pragma unroll
  for (int q = 0; q < 3; ++q) row[q] = -(c.x * RS[q] + c.y * RS[3 + q] + c.z * RS[6 + q]);
  row[3] = c.x; row[4] = c.y; row[5] = c.z;
  float rx, ry, rz;
  odom_qmul_vec(tf.qx, tf.qy, tf.qz, tf.qw, p.x, p.y, p.z, rx, ry, rz);
  d2 = c.x * (rx + tf.px) + c.y * (ry + tf.py) + c.z * (rz + tf.pz) + c.w;
}

// cyclic Jacobi eigen-decomposition of a symmetric 6x6 (float), ascending eigenvalues, vectors in columns.  Everything but
// the sweep loop is unrolled with compile-time indices so that A and V live in registers (one thread runs this on the
// critical path of the LaserOdom chain); the operation order is the oracle's.
__device__ __forceinline__ void sym_eigen6(const float *Ain, float *evals, float *V) {
  float A[36];
#pragma unroll
  for (int i = 0; i < 36; ++i) { A[i] = Ain[i]; V[i] = (i % 7 == 0) ? 1.f : 0.f; }
#pragma unroll 1
  for (int sweep = 0; sweep < 60; ++sweep) {
    float off = 0.f, diag = 0.f;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      diag += A[i * 6 + i] * A[i * 6 + i];
#pragma unroll
      for (int j = i + 1; j < 6; ++j) off += A[i * 6 + j] * A[i * 6 + j];
    }
    if (off <= FLT_EPSILON * FLT_EPSILON * diag || off == 0.f) break;
#pragma unroll
    for (int p = 0; p < 5; ++p)
#pragma unroll
      for (int q = p + 1; q < 6; ++q) {
        const float apq = A[p * 6 + q];
        if (apq != 0.f) {
          const float theta = (A[q * 6 + q] - A[p * 6 + p]) / (2.f * apq);
          const float t = (theta >= 0.f ? 1.f : -1.f) / (fabsf(theta) + sqrtf(theta * theta + 1.f));
          const float c = 1.f / sqrtf(t * t + 1.f), s = t * c;
#pragma unroll
          for (int k = 0; k < 6; ++k) { float a = A[k * 6 + p], b = A[k * 6 + q]; A[k * 6 + p] = c * a - s * b; A[k * 6 + q] = s * a + c * b; }
#pragma unroll
          for (int k = 0; k < 6; ++k) { float a = A[p * 6 + k], b = A[q * 6 + k]; A[p * 6 + k] = c * a - s * b; A[q * 6 + k] = s * a + c * b; }
#pragma unroll
          for (int k = 0; k < 6; ++k) { float a = V[k * 6 + p], b = V[k * 6 + q]; V[k * 6 + p] = c * a - s * b; V[k * 6 + q] = s * a + c * b; }
        }
      }
  }
  // ascending order of the diagonal by the same exchange sort on an index array (first index wins ties)
  float d[6];
  int idx[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) { d[i] = A[i * 6 + i]; idx[i] = i; }
#pragma unroll
  for (int i = 0; i < 5; ++i)
#pragma unroll
    for (int j = i + 1; j < 6; ++j)
      if (d[j] < d[i]) { const float td = d[i]; d[i] = d[j]; d[j] = td; const int ti = idx[i]; idx[i] = idx[j]; idx[j] = ti; }
  float Vc[36];
#pragma unroll
  for (int i = 0; i < 36; ++i) Vc[i] = V[i];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    evals[j] = d[j];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      float v = Vc[k * 6];
#pragma unroll
      for (int c = 1; c < 6; ++c) v = (idx[j] == c) ? Vc[k * 6 + c] : v;
      V[k * 6 + j] = v;
    }
  }
}

// round < 0: CalculateLaserOdom (the first executed round carries the degeneracy analysis);  round >= 0: scan-to-map loop
// index of PointMapping::OptimizeTransformTobeMapped, where a round with fewer than min_features matches is skipped
// entirely (`continue`, PointMapping.cc:609-611) and the degeneracy analysis belongs to loop index 0 only.
__device__ inline void odom_solve_step(OdomState *__restrict__ st, TransformF *__restrict__ tf_dev, double delta_r_abort, double delta_t_abort,
                                int round = -1, const int *__restrict__ n_dev = nullptr, int min_features = 0, int left_update = 0,
                                float eig_thre = 100.f) {
  if (n_dev && *n_dev < min_features) { st->iter += 1; return; }
  const bool first_round = round < 0 ? (st->iter == 0) : (round == 0);
  float A[6][6], B[6], X[6], AtA[36];
  for (int a = 0; a < 6; ++a) { for (int b = 0; b < 6; ++b) { A[a][b] = (float)st->AtA[a * 6 + b]; AtA[a * 6 + b] = A[a][b]; } B[a] = (float)st->AtB[a]; }
  colpiv_qr_solve<6, 6>(A, B, X);
  if (first_round) {
    float E[6], V[36], V2[36];
    sym_eigen6(AtA, E, V);
    for (int k = 0; k < 36; ++k) V2[k] = V[k];
    int degenerate = 0;
    for (int i = 0; i < 6; ++i) {
      if (E[i] < eig_thre) { for (int j = 0; j < 6; ++j) V2[i * 6 + j] = 0.f; degenerate = 1; }
      else break;
    }
    for (int a = 0; a < 6; ++a)
      for (int c = 0; c < 6; ++c) { float s = 0.f; for (int k = 0; k < 6; ++k) s += V2[a * 6 + k] * V[c * 6 + k]; st->matP[a * 6 + c] = s; }
    st->degenerate = degenerate;
  }
  if (st->degenerate) {
    float X2[6];
    for (int a = 0; a < 6; ++a) { float s = 0.f; for (int c = 0; c < 6; ++c) s += st->matP[a * 6 + c] * X[c]; X2[a] = s; }
    for (int a = 0; a < 6; ++a) X[a] = X2[a];
  }
  TransformF tf = *tf_dev;
  // R_SO3(local_transform.rot): normalised copy of the rotation before the update
  float n0 = sqrtf(tf.qx * tf.qx + tf.qy * tf.qy + tf.qz * tf.qz + tf.qw * tf.qw);
  float ox = tf.qx / n0, oy = tf.qy / n0, oz = tf.qz / n0, ow = tf.qw / n0;
  tf.px += X[3]; tf.py += X[4]; tf.pz += X[5];
  {  // rot = rot * DeltaQ(X[0..2])  (Hamilton product, not normalised)
    float dx = X[0] / 2.f, dy = X[1] / 2.f, dz = X[2] / 2.f, dw = 1.f;
    float nw, nx, ny, nz;
    if (left_update) {  // rot = DeltaQ(x) * rot  (MapBuilder.cc:984-985)
      nw = dw * tf.qw - dx * tf.qx - dy * tf.qy - dz * tf.qz;
      nx = dw * tf.qx + dx * tf.qw + dy * tf.qz - dz * tf.qy;
      ny = dw * tf.qy + dy * tf.qw + dz * tf.qx - dx * tf.qz;
      nz = dw * tf.qz + dz * tf.qw + dx * tf.qy - dy * tf.qx;
    } else {
      nw = tf.qw * dw - tf.qx * dx - tf.qy * dy - tf.qz * dz;
      nx = tf.qw * dx + tf.qx * dw + tf.qy * dz - tf.qz * dy;
      ny = tf.qw * dy + tf.qy * dw + tf.qz * dx - tf.qx * dz;
      nz = tf.qw * dz + tf.qz * dw + tf.qx * dy - tf.qy * dx;
    }
    tf.qx = nx; tf.qy = ny; tf.qz = nz; tf.qw = nw;
  }
  if (!isfinite(tf.px)) tf.px = 0.f;
  if (!isfinite(tf.py)) tf.py = 0.f;
  if (!isfinite(tf.pz)) tf.pz = 0.f;
  *tf_dev = tf;
  // angularDistance: d = a * b.conjugate(); 2*atan2(|d.vec|, |d.w|)
  float cw = ow * tf.qw + ox * tf.qx + oy * tf.qy + oz * tf.qz;
  float cx = -ow * tf.qx + ox * tf.qw - oy * tf.qz + oz * tf.qy;
  float cy = -ow * tf.qy + oy * tf.qw - oz * tf.qx + ox * tf.qz;
  float cz = -ow * tf.qz + oz * tf.qw - ox * tf.qy + oy * tf.qx;
  float ad = 2.f * atan2f(sqrtf(cx * cx + cy * cy + cz * cz), fabsf(cw));
  float delta_r = (float)((double)ad * 180.0 / M_PI);
  double tx = (double)(X[3] * 100.f), ty = (double)(X[4] * 100.f), tz = (double)(X[5] * 100.f);
  float delta_t = (float)sqrt(tx * tx + ty * ty + tz * tz);
  st->iter += 1;
  if ((double)delta_r < delta_r_abort && (double)delta_t < delta_t_abort) st->done = 1;
}


}  // namespace lio
