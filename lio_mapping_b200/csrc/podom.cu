// lio::PointOdometry - the scan-to-scan odometry of the pre-initialisation phase and the /compact_data pass-through that is
// left of it once the estimator switches it off - SURVEY section 8 row f4.  Reference: src/point_processor/PointOdometry.cc
//   TransformToStart / TransformToEnd      :237-292
//   Process                                :294-708   first sweep :302-310; per iteration (<= 25): corner matching :338-441
//                                                     (nearest point + nearest point of a neighbouring ring, searched every
//                                                     5th iteration), surf matching :443-549 (nearest + same-or-lower ring +
//                                                     higher ring), 6 x 6 float Gauss-Newton with the 0.1 step damping
//                                                     :551-664; transform_sum_ :667-669; de-skew + swap :673-690
//   PublishResults                         :710-766   io_ratio gate, TransformToEnd(full_cloud_), /compact_data payload
// Device design: the last clouds are a few ten thousand points (<= 1 MB, L2 resident) and the queries a few thousand, so the
// nearest-neighbour search is an exact brute-force scan - one CTA per 8 queries, every loaded point tested against all 8,
// (d2, index) packed into one 64-bit key so that min() gives the kd-tree's answer with ties by index - followed by a
// warp-per-query scan of the neighbouring rings that reproduces the sequential "first strictly smaller wins" rule through a
// (d2, visit order) key.  One iteration = one single-CTA kernel: TransformToStart of every query, the line / plane
// coefficients from the stored indices, the 6 x 6 normal equations (float products accumulated in double, fixed tree),
// colPivHouseholderQr solve, the first-iteration degeneracy projection and the convergence test; the iteration chain is
// enqueued once and later rounds return at once when the state says converged.  Pose compositions happen once per sweep on the
// host in the reference's float order (twistf.h).  Compiled with -fmad=false.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include "odom.cuh"
#include "twistf.h"

namespace lio {

constexpr int kPoQ = 8;            // queries per search CTA
constexpr int kPoSearchThreads = 256;
constexpr int kPoRoundThreads = 256;
constexpr unsigned kPoDown = 1u << 30;   // visit-order offset of the downward ring scan

// q_s = identity.slerp(s, q_e) (Eigen QuaternionBase::slerp), conjugated: the rotation TransformToStart / TransformToEnd apply
__device__ __forceinline__ void po_slerp_conj(const TransformF &es, float s, float &cx, float &cy, float &cz, float &cw) {
  const float one = 1.0f - FLT_EPSILON;
  const float d = es.qw;
  const float absD = fabsf(d);
  float scale0, scale1;
  if (absD >= one) { scale0 = 1.0f - s; scale1 = s; }
  else {
    const float theta = acosf(absD);
    const float sinTheta = sinf(theta);
    scale0 = sinf((1.0f - s) * theta) / sinTheta;
    scale1 = sinf(s * theta) / sinTheta;
  }
  if (d < 0.f) scale1 = -scale1;
  cw = scale0 * 1.0f + scale1 * es.qw;
  cx = -(scale0 * 0.0f + scale1 * es.qx); cy = -(scale0 * 0.0f + scale1 * es.qy); cz = -(scale0 * 0.0f + scale1 * es.qz);
}

// PointOdometry::TransformToStart :237-259
__device__ __forceinline__ float4 po_to_start(float4 pi, const TransformF &es, float time_factor) {
  const float s = time_factor * (pi.w - (float)(int)pi.w);
  if (s < 0 || (double)s > 1.001) return pi;
  const float x = pi.x - s * es.px, y = pi.y - s * es.py, z = pi.z - s * es.pz;
  float cx, cy, cz, cw;
  po_slerp_conj(es, s, cx, cy, cz, cw);
  float4 po;
  odom_qmul_vec(cx, cy, cz, cw, x, y, z, po.x, po.y, po.z);
  po.w = pi.w;
  return po;
}

// PointOdometry::TransformToEnd :261-292, in place, on *n_dev points with transform_es_ from the device.  normalise: the
// rotation normalised first (transform_es_.rot.normalize() :675, the host's float expression), as the full cloud of
// PublishResults sees it.
__global__ void __launch_bounds__(256) po_to_end(float4 *__restrict__ cloud, const int *__restrict__ n_dev, const TransformF *__restrict__ tf_dev,
                                                 int normalise, float time_factor) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *n_dev) return;
  TransformF es = *tf_dev;
  if (normalise) {
    const float n = sqrtf(es.qx * es.qx + es.qy * es.qy + es.qz * es.qz + es.qw * es.qw);
    es.qx /= n; es.qy /= n; es.qz /= n; es.qw /= n;
  }
  float4 p = cloud[i];
  const float s = time_factor * (p.w - (float)(int)p.w);
  p.x -= s * es.px; p.y -= s * es.py; p.z -= s * es.pz;
  p.w = (float)(int)p.w;
  float cx, cy, cz, cw;
  po_slerp_conj(es, s, cx, cy, cz, cw);
  float ax, ay, az, bx, by, bz;
  odom_qmul_vec(cx, cy, cz, cw, p.x, p.y, p.z, ax, ay, az);
  odom_qmul_vec(es.qx, es.qy, es.qz, es.qw, ax, ay, az, bx, by, bz);
  cloud[i] = make_float4(bx + es.px, by + es.py, bz + es.pz, p.w);
}

// Ingest of the device entry: the five counts read on the device and clamped to their bounds into cnt[0..4], and the
// clouds that outlive the call (less sharp, less flat, full: blockIdx.y 0..2) copied into the context's buffers.
struct PoIngest {
  const float4 *src[3];
  float4 *dst[3];
  const int *n_in[5];
  int n_max[5];
};
__global__ void __launch_bounds__(256) po_ingest(PoIngest a, int *__restrict__ cnt) {
  const int y = blockIdx.y;
  const int k = y == 0 ? 1 : (y == 1 ? 3 : 4);   // count slot of the copied cloud
  int n = *a.n_in[k];
  n = n < 0 ? 0 : (n > a.n_max[k] ? a.n_max[k] : n);
  if (blockIdx.x == 0 && y == 0 && threadIdx.x < 5) {
    const int j = threadIdx.x;
    const int v = *a.n_in[j];
    cnt[j] = v < 0 ? 0 : (v > a.n_max[j] ? a.n_max[j] : v);
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) a.dst[y][i] = __ldg(a.src[y] + i);
}

__device__ __forceinline__ unsigned long long po_min64(unsigned long long a, unsigned long long b) { return a < b ? a : b; }
__device__ __forceinline__ unsigned long long po_warp_min(unsigned long long v) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) v = po_min64(v, __shfl_xor_sync(0xffffffffu, v, off));
  return v;
}
__device__ __forceinline__ float po_sqdiff(float4 a, float4 b) {   // CalcSquaredDiff(a, b), math_utils.h:85-91
  const float dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z;
  return dx * dx + dy * dy + dz * dz;
}
__device__ __forceinline__ int po_visit_to_index(unsigned v, int c) { return v < kPoDown ? c + 1 + (int)v : c - 1 - (int)(v - kPoDown); }

// KIND 0: corner_points_sharp_ against last_corner_cloud_ (2 indices per query); KIND 1: surf_points_flat_ against
// last_surf_cloud_ (3 indices per query).
template <int KIND>
__global__ void __launch_bounds__(kPoSearchThreads)
po_search(const float4 *__restrict__ query, const int *__restrict__ nq_dev, const float4 *__restrict__ last, int nlast,
          const TransformF *__restrict__ tf_dev, const OdomState *__restrict__ st, float time_factor, int *__restrict__ idx_out) {
  const int nq = *nq_dev;   // the grid covers the bound; CTAs past the count leave at once
  if (st->done || (int)blockIdx.x * kPoQ >= nq) return;
  __shared__ float4 s_sel[kPoQ];
  __shared__ unsigned long long s_best[kPoSearchThreads / 32][kPoQ];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int q0 = blockIdx.x * kPoQ;
  const TransformF es = *tf_dev;
  if (tid < kPoQ) {
    const int qi = q0 + tid;
    s_sel[tid] = qi < nq ? po_to_start(__ldg(query + qi), es, time_factor) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  float sx[kPoQ], sy[kPoQ], sz[kPoQ];
  unsigned long long best[kPoQ];
#pragma unroll
  for (int q = 0; q < kPoQ; ++q) { const float4 s = s_sel[q]; sx[q] = s.x; sy[q] = s.y; sz[q] = s.z; best[q] = ~0ull; }
  for (int j = tid; j < nlast; j += kPoSearchThreads) {
    const float4 p = __ldg(last + j);
#pragma unroll
    for (int q = 0; q < kPoQ; ++q) {
      const float dx = p.x - sx[q], dy = p.y - sy[q], dz = p.z - sz[q];
      const float d2 = dx * dx + dy * dy + dz * dz;
      best[q] = po_min64(best[q], ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)j);
    }
  }
#pragma unroll
  for (int q = 0; q < kPoQ; ++q) {
    const unsigned long long b = po_warp_min(best[q]);
    if (lane == 0) s_best[warp][q] = b;
  }
  __syncthreads();
  // warp w finishes query w: nearest point, then the ring scans
  const int qi = q0 + warp;
  if (warp >= kPoQ || qi >= nq) return;
  const unsigned long long key = po_warp_min(lane < kPoSearchThreads / 32 ? s_best[lane][warp] : ~0ull);
  const float d2min = __uint_as_float((unsigned)(key >> 32));
  constexpr int NI = KIND == 0 ? 2 : 3;
  if (!(d2min < 25.f)) {
    if (lane < NI) idx_out[NI * qi + lane] = -1;
    return;
  }
  const int c = (int)(unsigned)(key & 0xffffffffu);
  const float4 sel = s_sel[warp];
  const int scan = (int)__ldg(last + c).w;
  unsigned long long k2 = ~0ull, k3 = ~0ull;   // KIND 0 uses k2 only
  // upward: j = c + 1 ..., stop at the first ring > scan + 2.5
  for (int base = c + 1; base < nlast; base += 32) {
    const int j = base + lane;
    const bool valid = j < nlast;
    const float4 p = valid ? __ldg(last + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int ring = (int)p.w;
    const bool brk = valid && ((double)ring > (double)scan + 2.5);
    const unsigned bm = __ballot_sync(0xffffffffu, brk);
    const int first = bm ? __ffs(bm) - 1 : 32;
    if (valid && lane < first) {
      const float d2 = po_sqdiff(p, sel);
      if (d2 < 25.f) {
        const unsigned long long k = ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)(j - c - 1);
        if (KIND == 0) { if (ring > scan) k2 = po_min64(k2, k); }
        else { if (ring <= scan) k2 = po_min64(k2, k); else k3 = po_min64(k3, k); }
      }
    }
    if (bm) break;
  }
  // downward: j = c - 1 ..., stop at the first ring < scan - 2.5
  for (int base = c - 1; base >= 0; base -= 32) {
    const int j = base - lane;
    const bool valid = j >= 0;
    const float4 p = valid ? __ldg(last + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int ring = (int)p.w;
    const bool brk = valid && ((double)ring < (double)scan - 2.5);
    const unsigned bm = __ballot_sync(0xffffffffu, brk);
    const int first = bm ? __ffs(bm) - 1 : 32;
    if (valid && lane < first) {
      const float d2 = po_sqdiff(p, sel);
      if (d2 < 25.f) {
        const unsigned long long k = ((unsigned long long)__float_as_uint(d2) << 32) | (kPoDown + (unsigned)(c - 1 - j));
        if (KIND == 0) { if (ring < scan) k2 = po_min64(k2, k); }
        else { if (ring >= scan) k2 = po_min64(k2, k); else k3 = po_min64(k3, k); }
      }
    }
    if (bm) break;
  }
  k2 = po_warp_min(k2);
  if (KIND == 1) k3 = po_warp_min(k3);
  if (lane == 0) {
    idx_out[NI * qi] = c;
    idx_out[NI * qi + 1] = k2 == ~0ull ? -1 : po_visit_to_index((unsigned)(k2 & 0xffffffffu), c);
    if (KIND == 1) idx_out[NI * qi + 2] = k3 == ~0ull ? -1 : po_visit_to_index((unsigned)(k3 & 0xffffffffu), c);
  }
}

// One iteration of the loop :333-664 after the searches: coefficients, normal equations, solve, update, convergence.
__global__ void __launch_bounds__(kPoRoundThreads)
po_round(const float4 *__restrict__ sharp, const float4 *__restrict__ flat, const int *__restrict__ counts, const float4 *__restrict__ last_corner,
         const float4 *__restrict__ last_surf, const int *__restrict__ idx_c, const int *__restrict__ idx_s, TransformF *__restrict__ tf_dev,
         OdomState *__restrict__ st, float time_factor, int iter, int *__restrict__ nsel_out) {
  if (st->done) return;
  const int ns = counts[0], nf = counts[2];   // sharp, flat
  __shared__ double s_red[kPoRoundThreads / 32][28];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const TransformF es = *tf_dev;
  float R[9];
  odom_rotation(es, R);
  double acc[27];
#pragma unroll
  for (int k = 0; k < 27; ++k) acc[k] = 0.0;
  int cnt = 0;
  for (int i = tid; i < ns + nf; i += kPoRoundThreads) {
    const bool corner = i < ns;
    const float4 pi = corner ? __ldg(sharp + i) : __ldg(flat + (i - ns));
    const float4 sel = po_to_start(pi, es, time_factor);
    float4 coeff = make_float4(0.f, 0.f, 0.f, 0.f);
    bool accept = false;
    if (corner) {
      const int i1 = idx_c[2 * i], i2 = idx_c[2 * i + 1];
      if (i2 >= 0) {
        const float4 t1 = __ldg(last_corner + i1), t2 = __ldg(last_corner + i2);
        const float x0 = sel.x, y0 = sel.y, z0 = sel.z, x1 = t1.x, y1 = t1.y, z1 = t1.z, x2 = t2.x, y2 = t2.y, z2 = t2.z;
        const float mxy = (x0 - x1) * (y0 - y2) - (x0 - x2) * (y0 - y1);
        const float mxz = (x0 - x1) * (z0 - z2) - (x0 - x2) * (z0 - z1);
        const float myz = (y0 - y1) * (z0 - z2) - (y0 - y2) * (z0 - z1);
        const float a012 = sqrtf(mxy * mxy + mxz * mxz + myz * myz);
        const float l12 = sqrtf((x1 - x2) * (x1 - x2) + (y1 - y2) * (y1 - y2) + (z1 - z2) * (z1 - z2));
        const float la = ((y1 - y2) * mxy + (z1 - z2) * mxz) / a012 / l12;
        const float lb = -((x1 - x2) * mxy - (z1 - z2) * myz) / a012 / l12;
        const float lc = -((x1 - x2) * mxz + (y1 - y2) * myz) / a012 / l12;
        const float ld2 = a012 / l12;
        float s = 1;
        if (iter >= 5) s = 1 - 1.8f * fabsf(ld2);
        coeff = make_float4(s * la, s * lb, s * lc, s * ld2);
        accept = (double)s > 0.1 && ld2 != 0;
      }
    } else {
      const int q = i - ns;
      const int i1 = idx_s[3 * q], i2 = idx_s[3 * q + 1], i3 = idx_s[3 * q + 2];
      if (i2 >= 0 && i3 >= 0) {
        const float4 t1 = __ldg(last_surf + i1), t2 = __ldg(last_surf + i2), t3 = __ldg(last_surf + i3);
        float pa = (t2.y - t1.y) * (t3.z - t1.z) - (t3.y - t1.y) * (t2.z - t1.z);
        float pb = (t2.z - t1.z) * (t3.x - t1.x) - (t3.z - t1.z) * (t2.x - t1.x);
        float pc = (t2.x - t1.x) * (t3.y - t1.y) - (t3.x - t1.x) * (t2.y - t1.y);
        float pd = -(pa * t1.x + pb * t1.y + pc * t1.z);
        const float ps = sqrtf(pa * pa + pb * pb + pc * pc);
        pa /= ps; pb /= ps; pc /= ps; pd /= ps;
        const float pd2 = pa * sel.x + pb * sel.y + pc * sel.z + pd;
        float s = 1;
        if (iter >= 5) s = 1 - 1.8f * fabsf(pd2) / sqrtf(sqrtf(sel.x * sel.x + sel.y * sel.y + sel.z * sel.z));
        coeff = make_float4(s * pa, s * pb, s * pc, s * pd2);
        accept = (double)s > 0.1 && pd2 != 0;
      }
    }
    if (accept) {
      ++cnt;
      // J_r = w^T [rot^* (p - t)]x, J_t = -w^T R^T, rhs -0.1 d2   (:566-587)
      float vx, vy, vz;
      odom_qmul_vec(-es.qx, -es.qy, -es.qz, es.qw, pi.x - es.px, pi.y - es.py, pi.z - es.pz, vx, vy, vz);
      float row[6];
      row[0] = coeff.x * 0.f + coeff.y * vz + coeff.z * (-vy);
      row[1] = coeff.x * (-vz) + coeff.y * 0.f + coeff.z * vx;
      row[2] = coeff.x * vy + coeff.y * (-vx) + coeff.z * 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) row[3 + c] = (-coeff.x) * R[c * 3 + 0] + (-coeff.y) * R[c * 3 + 1] + (-coeff.z) * R[c * 3 + 2];
      const float b = (float)(-0.1 * (double)coeff.w);
      int k = 0;
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int c = a; c < 6; ++c) acc[k++] += (double)(row[a] * row[c]);
#pragma unroll
      for (int a = 0; a < 6; ++a) acc[21 + a] += (double)(row[a] * b);
    }
  }
#pragma unroll
  for (int k = 0; k < 27; ++k) {
    double v = acc[k];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) s_red[warp][k] = v;
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
  if (lane == 0) s_red[warp][27] = (double)cnt;
  __syncthreads();
  if (tid < 28) {
    double v = 0.0;
    for (int w = 0; w < kPoRoundThreads / 32; ++w) v += s_red[w][tid];
    s_red[0][tid] = v;
  }
  __syncthreads();
  if (tid == 0) {
    int k = 0;
    for (int a = 0; a < 6; ++a)
      for (int c = a; c < 6; ++c) { st->AtA[a * 6 + c] = s_red[0][k]; st->AtA[c * 6 + a] = s_red[0][k]; ++k; }
    for (int a = 0; a < 6; ++a) st->AtB[a] = s_red[0][21 + a];
    *nsel_out = (int)s_red[0][27];
    odom_solve_step(st, tf_dev, 0.1, 0.1, iter, nsel_out, 10, 0, 10.f);   // num_point_sel < 10 -> continue; abort 0.1 deg / 0.1 cm
  }
}

}  // namespace lio

using namespace lio;

// Pinned staging of one process call: what goes up (start pose, host-path counts) and the single read-back.
struct PoStage {
  TransformF tf_up;
  int cnt_up[5];
  int cnt[5];      // sharp, less_sharp, flat, less_flat, full as the kernels saw them (clamped)
  int iter, nsel;
  TransformF tf;
};

struct lio_po {
  int device = 0;
  cudaStream_t stream = nullptr;
  float time_factor = 10.f;
  int io_ratio = 2, max_iter = 25;
  int cap_feat = 0, cap_full = 0;
  bool system_inited = false, enable_odom = true;
  long frame_count = 0;
  float4 *d_sharp = nullptr, *d_flat = nullptr, *d_less_sharp = nullptr, *d_less_flat = nullptr, *d_last_corner = nullptr, *d_last_surf = nullptr,
         *d_full = nullptr;
  int n_sharp = 0, n_flat = 0, n_less_sharp = 0, n_less_flat = 0, n_last_corner = 0, n_last_surf = 0, n_full = 0;   // host copies (read-back)
  // device counts of the last call: [0] sharp [1] less_sharp (now last_corner) [2] flat [3] less_flat (now last_surf) [4] full;
  // [7] stays 0 (the count of an absent cloud)
  int *d_cnt = nullptr;
  int *d_idx_c = nullptr, *d_idx_s = nullptr, *d_nsel = nullptr;
  TransformF *d_tf = nullptr;
  OdomState *d_odom = nullptr;
  PoStage *h_stage = nullptr;
  TwistF es, sum;
  int published = 0;
  int launches = 0;
  CallStats stats;
};

extern "C" int lio_po_destroy(lio_po *p) {
  if (!p) return LIO_OK;
  cudaSetDevice(p->device);
  void *fr[] = {p->d_sharp, p->d_flat, p->d_less_sharp, p->d_less_flat, p->d_last_corner, p->d_last_surf, p->d_full, p->d_cnt, p->d_idx_c,
                p->d_idx_s, p->d_nsel, p->d_tf, p->d_odom};
  for (void *q : fr) if (q) cudaFree(q);
  if (p->h_stage) cudaFreeHost(p->h_stage);
  delete p;
  return LIO_OK;
}

extern "C" int lio_po_create(float scan_period, int io_ratio, int num_max_iterations, int max_feature_points, int max_full_points, int device,
                             void *cuda_stream, lio_po **out) {
  if (!out || !(scan_period > 0) || num_max_iterations < 0 || max_feature_points < 16 || max_full_points < 16) return LIO_ERR_INVALID;
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  LIO_CUDA_OK(cudaSetDevice(device));
  lio_po *p = new (std::nothrow) lio_po();
  if (!p) return LIO_ERR_INVALID;
  p->device = device; p->stream = (cudaStream_t)cuda_stream;
  p->time_factor = 1 / scan_period; p->io_ratio = io_ratio; p->max_iter = num_max_iterations;
  p->cap_feat = max_feature_points; p->cap_full = max_full_points;
  bool ok = true;
  float4 **clouds[] = {&p->d_sharp, &p->d_flat, &p->d_less_sharp, &p->d_less_flat, &p->d_last_corner, &p->d_last_surf};
  for (float4 **c : clouds) ok = ok && cudaMalloc(c, sizeof(float4) * max_feature_points) == cudaSuccess;
  ok = ok && cudaMalloc(&p->d_full, sizeof(float4) * max_full_points) == cudaSuccess;
  ok = ok && cudaMalloc(&p->d_cnt, sizeof(int) * 8) == cudaSuccess && cudaMemset(p->d_cnt, 0, sizeof(int) * 8) == cudaSuccess;
  ok = ok && cudaMalloc(&p->d_idx_c, sizeof(int) * 2 * max_feature_points) == cudaSuccess;
  ok = ok && cudaMalloc(&p->d_idx_s, sizeof(int) * 3 * max_feature_points) == cudaSuccess;
  ok = ok && cudaMalloc(&p->d_nsel, sizeof(int)) == cudaSuccess;
  ok = ok && cudaMalloc(&p->d_tf, sizeof(TransformF)) == cudaSuccess;
  ok = ok && cudaMalloc(&p->d_odom, sizeof(OdomState)) == cudaSuccess;
  ok = ok && cudaMallocHost(&p->h_stage, sizeof(PoStage)) == cudaSuccess;
  if (!ok) { lio_set_last_error(__FILE__, __LINE__, "lio_po_create: device allocation failed"); lio_po_destroy(p); return LIO_ERR_CUDA; }
  *out = p;
  return LIO_OK;
}

extern "C" int lio_po_set_enable_odom(lio_po *p, int enable) {   // the /enable_odom service, PointOdometry.cc:126-131
  if (!p) return LIO_ERR_INVALID;
  p->enable_odom = enable > 0;
  return LIO_OK;
}

static void po_store(const TwistF &t, float *o) { o[0] = t.qx; o[1] = t.qy; o[2] = t.qz; o[3] = t.qw; o[4] = t.px; o[5] = t.py; o[6] = t.pz; }

// Process + PublishResults (:294-766) once the sweep is in place: less sharp / less flat / full in the context's buffers,
// the five clamped counts in d_cnt[0..4], sharp / flat at `sharp` / `flat` (the caller's buffers or the context's).  mx_*
// bound the counts and size the grids.  One synchronisation: the read-back of transform_es_, the iteration and match
// counts and the five counts, from which the host learns the sizes of the new "last" clouds (the :324 gate of the next call).
static int po_core(lio_po *p, const float4 *sharp, int mx_sharp, const float4 *flat, int mx_flat, int mx_less_sharp, int mx_less_flat, int mx_full,
                   float transform_sum7[7], float transform_es7[7], int info4[4]) {
  cudaStream_t st = p->stream;
  CallStats &S = p->stats;
  PoStage *h = p->h_stage;
  const float tfac = p->time_factor;
  const bool first = !p->system_inited;   // :302-310: the first sweep only becomes the last clouds
  bool solved = false;
  p->published = 0;
  auto to_end = [&](float4 *cloud, const int *n_dev, int n_max, int normalise) {
    if (n_max > 0) { po_to_end<<<(n_max + 255) / 256, 256, 0, st>>>(cloud, n_dev, p->d_tf, normalise, tfac); ++p->launches; }
  };
  if (first) {
    p->system_inited = true;
  } else {
    ++p->frame_count;
    if (p->enable_odom) {
      h->tf_up = TransformF{p->es.qx, p->es.qy, p->es.qz, p->es.qw, p->es.px, p->es.py, p->es.pz};
      LIO_CUDA_OK(stats_h2d(S, p->d_tf, &h->tf_up, sizeof(TransformF), st));
      if (p->n_last_corner > 10 && p->n_last_surf > 100) {   // :324
        LIO_CUDA_OK(cudaMemsetAsync(p->d_odom, 0, sizeof(OdomState), st));
        LIO_CUDA_OK(cudaMemsetAsync(p->d_nsel, 0, sizeof(int), st));
        for (int it = 0; it < p->max_iter; ++it) {
          if (it % 5 == 0) {
            if (mx_sharp) { po_search<0><<<(mx_sharp + kPoQ - 1) / kPoQ, kPoSearchThreads, 0, st>>>(sharp, p->d_cnt + 0, p->d_last_corner, p->n_last_corner, p->d_tf, p->d_odom, tfac, p->d_idx_c); ++p->launches; }
            if (mx_flat) { po_search<1><<<(mx_flat + kPoQ - 1) / kPoQ, kPoSearchThreads, 0, st>>>(flat, p->d_cnt + 2, p->d_last_surf, p->n_last_surf, p->d_tf, p->d_odom, tfac, p->d_idx_s); ++p->launches; }
          }
          po_round<<<1, kPoRoundThreads, 0, st>>>(sharp, flat, p->d_cnt, p->d_last_corner, p->d_last_surf, p->d_idx_c, p->d_idx_s, p->d_tf, p->d_odom, tfac,
                                                 it, p->d_nsel);
          ++p->launches;
        }
        solved = true;
      }
      // de-skew of the clouds that become the last ones (:673-674) with the unnormalised transform_es_
      to_end(p->d_less_sharp, p->d_cnt + 1, mx_less_sharp, 0);
      to_end(p->d_less_flat, p->d_cnt + 3, mx_less_flat, 0);
    }
    if (p->io_ratio < 2 || p->frame_count % p->io_ratio == 1) {   // PublishResults :726-765
      if (p->enable_odom) to_end(p->d_full, p->d_cnt + 4, mx_full, 1);
      p->published = 1;
    }
  }
  LIO_CUDA_OK(cudaGetLastError());
  LIO_CUDA_OK(stats_d2h(S, h->cnt, p->d_cnt, sizeof(h->cnt), st));
  if (solved) {
    LIO_CUDA_OK(stats_d2h(S, &h->tf, p->d_tf, sizeof(TransformF), st));
    LIO_CUDA_OK(stats_d2h(S, &h->iter, &p->d_odom->iter, sizeof(int), st));
    LIO_CUDA_OK(stats_d2h(S, &h->nsel, p->d_nsel, sizeof(int), st));
  }
  LIO_CUDA_OK(stats_sync(S, st));
  LIO_CUDA_OK(cudaGetLastError());
  S.launches = p->launches;
  p->n_sharp = h->cnt[0]; p->n_less_sharp = h->cnt[1]; p->n_flat = h->cnt[2]; p->n_less_flat = h->cnt[3]; p->n_full = h->cnt[4];
  int iters = 0, nsel = 0;
  if (solved) {
    p->es = TwistF{h->tf.qx, h->tf.qy, h->tf.qz, h->tf.qw, h->tf.px, h->tf.py, h->tf.pz};
    iters = h->iter; nsel = h->nsel;
  }
  if (!first && p->enable_odom) {
    p->sum = twist_mul(p->sum, twist_inverse(p->es));   // transform_sum_ = transform_sum_ * transform_es_.inverse()  :667-669
    const float n = std::sqrt(p->es.qx * p->es.qx + p->es.qy * p->es.qy + p->es.qz * p->es.qz + p->es.qw * p->es.qw);   // :675
    p->es.qx /= n; p->es.qy /= n; p->es.qz /= n; p->es.qw /= n;
  }
  // corner_points_less_sharp_.swap(last_corner_cloud_), surf_points_less_flat_.swap(last_surf_cloud_); the device counts stay in
  // d_cnt[1] / d_cnt[3]
  std::swap(p->d_less_sharp, p->d_last_corner); std::swap(p->n_less_sharp, p->n_last_corner);
  std::swap(p->d_less_flat, p->d_last_surf); std::swap(p->n_less_flat, p->n_last_surf);
  if (transform_sum7) po_store(p->sum, transform_sum7);
  if (transform_es7) po_store(p->es, transform_es7);
  if (info4) { info4[0] = iters; info4[1] = p->published; info4[2] = (int)p->frame_count; info4[3] = nsel; }
  return LIO_OK;
}

// Host arrays: uploaded into the context's buffers, then the same core.
extern "C" int lio_po_process_host(lio_po *p, const float *sharp, int n_sharp, const float *less_sharp, int n_less_sharp, const float *flat,
                                   int n_flat, const float *less_flat, int n_less_flat, const float *full, int n_full, float transform_sum7[7],
                                   float transform_es7[7], int info4[4]) {
  if (!p || n_sharp < 0 || n_less_sharp < 0 || n_flat < 0 || n_less_flat < 0 || n_full < 0 || (n_sharp && !sharp) || (n_less_sharp && !less_sharp) ||
      (n_flat && !flat) || (n_less_flat && !less_flat) || (n_full && !full))
    return LIO_ERR_INVALID;
  if (std::max(std::max(n_sharp, n_less_sharp), std::max(n_flat, n_less_flat)) > p->cap_feat || n_full > p->cap_full) {
    lio_set_last_error(__FILE__, __LINE__, "lio_po_process_host: a cloud exceeds the capacity given to lio_po_create");
    return LIO_ERR_CAPACITY;
  }
  LIO_CUDA_OK(cudaSetDevice(p->device));
  cudaStream_t st = p->stream;
  p->stats.reset(); p->launches = 0;
  const float *src[5] = {sharp, less_sharp, flat, less_flat, full};
  float4 *dst[5] = {p->d_sharp, p->d_less_sharp, p->d_flat, p->d_less_flat, p->d_full};
  const int cnt[5] = {n_sharp, n_less_sharp, n_flat, n_less_flat, n_full};
  for (int k = 0; k < 5; ++k) {
    if (cnt[k]) LIO_CUDA_OK(stats_h2d(p->stats, dst[k], src[k], sizeof(float4) * cnt[k], st));
    p->h_stage->cnt_up[k] = cnt[k];
  }
  LIO_CUDA_OK(stats_h2d(p->stats, p->d_cnt, p->h_stage->cnt_up, sizeof(p->h_stage->cnt_up), st));
  return po_core(p, p->d_sharp, n_sharp, p->d_flat, n_flat, n_less_sharp, n_less_flat, n_full, transform_sum7, transform_es7, info4);
}

// Device clouds: the counts are clamped on the device and the clouds that outlive the call are copied in (one kernel),
// sharp / flat are read where they are.
extern "C" int lio_po_process_dev(lio_po *p, const lio_dev_cloud clouds[5], float transform_sum7[7], float transform_es7[7], int info4[4]) {
  if (!p || !clouds) return LIO_ERR_INVALID;
  for (int k = 0; k < 5; ++k)
    if (clouds[k].n_max < 0 || (clouds[k].n_max > 0 && (!clouds[k].xyzi || !clouds[k].n_dev))) return LIO_ERR_INVALID;
  for (int k = 0; k < 5; ++k)
    if (clouds[k].n_max > (k == 4 ? p->cap_full : p->cap_feat)) {
      lio_set_last_error(__FILE__, __LINE__, "lio_po_process_dev: n_max exceeds the capacity given to lio_po_create");
      return LIO_ERR_CAPACITY;
    }
  LIO_CUDA_OK(cudaSetDevice(p->device));
  cudaStream_t st = p->stream;
  p->stats.reset(); p->launches = 0;
  PoIngest a;
  const int copied[3] = {1, 3, 4};
  float4 *dst[3] = {p->d_less_sharp, p->d_less_flat, p->d_full};
  int mx = 0;
  for (int y = 0; y < 3; ++y) {
    a.src[y] = reinterpret_cast<const float4 *>(clouds[copied[y]].xyzi);
    a.dst[y] = dst[y];
    mx = std::max(mx, clouds[copied[y]].n_max);
  }
  for (int k = 0; k < 5; ++k) {
    a.n_in[k] = clouds[k].n_max > 0 ? clouds[k].n_dev : p->d_cnt + 7;
    a.n_max[k] = clouds[k].n_max;
  }
  po_ingest<<<dim3(std::max(1, std::min((mx + 255) / 256, 4 * 148)), 3), 256, 0, st>>>(a, p->d_cnt);
  ++p->launches;
  return po_core(p, reinterpret_cast<const float4 *>(clouds[0].xyzi), clouds[0].n_max, reinterpret_cast<const float4 *>(clouds[2].xyzi),
                 clouds[2].n_max, clouds[1].n_max, clouds[3].n_max, clouds[4].n_max, transform_sum7, transform_es7, info4);
}

extern "C" int lio_po_cloud_dev(lio_po *p, int which, const float **xyzi, const int **n_dev) {
  if (!p || !xyzi || !n_dev) return LIO_ERR_INVALID;
  switch (which) {
    case 0: *xyzi = reinterpret_cast<const float *>(p->d_last_corner); *n_dev = p->d_cnt + 1; return LIO_OK;
    case 1: *xyzi = reinterpret_cast<const float *>(p->d_last_surf); *n_dev = p->d_cnt + 3; return LIO_OK;
    case 2: *xyzi = reinterpret_cast<const float *>(p->d_full); *n_dev = p->d_cnt + 4; return LIO_OK;
    default: return LIO_ERR_INVALID;
  }
}

extern "C" int lio_po_last_stats(lio_po *p, long long out[4]) {
  if (!p || !out) return LIO_ERR_INVALID;
  out[0] = p->stats.launches; out[1] = p->stats.syncs; out[2] = p->stats.h2d; out[3] = p->stats.d2h;
  return LIO_OK;
}

static int po_cloud(lio_po *p, int which, const float4 **d, int *n) {
  switch (which) {
    case 0: *d = p->d_last_corner; *n = p->n_last_corner; return LIO_OK;
    case 1: *d = p->d_last_surf; *n = p->n_last_surf; return LIO_OK;
    case 2: *d = p->d_full; *n = p->n_full; return LIO_OK;
    default: return LIO_ERR_INVALID;
  }
}

extern "C" int lio_po_cloud_size(lio_po *p, int which, int *n) {
  const float4 *d;
  if (!p || !n) return LIO_ERR_INVALID;
  return po_cloud(p, which, &d, n);
}

extern "C" int lio_po_cloud_download(lio_po *p, int which, float *out_xyzi, int cap) {
  const float4 *d;
  int n = 0;
  if (!p || !out_xyzi) return LIO_ERR_INVALID;
  if (po_cloud(p, which, &d, &n) != LIO_OK) return LIO_ERR_INVALID;
  if (n > cap) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(p->device));
  if (n) LIO_CUDA_OK(cudaMemcpyAsync(out_xyzi, d, sizeof(float4) * n, cudaMemcpyDeviceToHost, p->stream));
  LIO_CUDA_OK(cudaStreamSynchronize(p->stream));
  return LIO_OK;
}

// the /compact_data payload of the sweep just processed (:732-762): 3 header points, then corner || surf || full
extern "C" int lio_po_compact_data(lio_po *p, float *out_xyzi, int cap_points, int *n_points) {
  if (!p || !out_xyzi || !n_points) return LIO_ERR_INVALID;
  if (!p->published) { lio_set_last_error(__FILE__, __LINE__, "lio_po_compact_data: the last sweep was not published (io_ratio gate or first sweep)"); return LIO_ERR_INVALID; }
  const int total = 3 + p->n_last_corner + p->n_last_surf + p->n_full;
  *n_points = total;
  if (total > cap_points) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(p->device));
  float *o = out_xyzi;
  o[0] = p->sum.px; o[1] = p->sum.py; o[2] = p->sum.pz; o[3] = 0.f;
  o[4] = p->sum.qx; o[5] = p->sum.qy; o[6] = p->sum.qz; o[7] = p->sum.qw;
  o[8] = (float)p->n_last_corner; o[9] = (float)p->n_last_surf; o[10] = (float)p->n_full; o[11] = p->sum.qw;   // the reused PointT keeps intensity
  o += 12;
  const float4 *src[3] = {p->d_last_corner, p->d_last_surf, p->d_full};
  const int cnt[3] = {p->n_last_corner, p->n_last_surf, p->n_full};
  for (int k = 0; k < 3; ++k) {
    if (cnt[k]) LIO_CUDA_OK(cudaMemcpyAsync(o, src[k], sizeof(float4) * cnt[k], cudaMemcpyDeviceToHost, p->stream));
    o += 4 * (size_t)cnt[k];
  }
  LIO_CUDA_OK(cudaStreamSynchronize(p->stream));
  return LIO_OK;
}

extern "C" int lio_po_last_launches(lio_po *p) { return p ? p->launches : 0; }

// test aid: the match indices of the last search (kind 0: 2 per sharp point, kind 1: 3 per flat point)
extern "C" int lio_po_matches(lio_po *p, int kind, int32_t *out, int cap_queries) {
  if (!p || !out || (kind != 0 && kind != 1)) return LIO_ERR_INVALID;
  const int nq = kind == 0 ? p->n_sharp : p->n_flat, per = kind == 0 ? 2 : 3;
  if (nq > cap_queries) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(p->device));
  if (nq) LIO_CUDA_OK(cudaMemcpy(out, kind == 0 ? p->d_idx_c : p->d_idx_s, sizeof(int) * per * nq, cudaMemcpyDeviceToHost));
  return LIO_OK;
}
