// lio::Estimator (steady state) on sm_100a — the host shell keeps the reference's control flow
// (window bookkeeping, gates, slide; src/imu_processor/Estimator.cc) while every per-point /
// per-feature loop runs in the CUDA kernels of this library:
//   ProcessLaserOdom INITED branch :618-774 -> process_scan   (de-skew kernel, device VoxelGrid)
//   BuildLocalMap :1361-1646                -> build_local_map (concat+transform kernel, VoxelGrid, cell hash,
//                                              voxel-hash kNN + plane fit per frame, device LaserOdom chain)
//   SolveOptimization :1648-2438            -> solve_optimization (fused residual+Jacobian+J^T J kernel per
//                                              iteration, dogleg controller, marginalisation)
//   SlideWindow :2570-2666                  -> slide_window
// There is no CPU path for the per-point work: without a CUDA device create() fails.
#include "assemble.cuh"
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include "factors_host.h"
#include "factors_impl.h"
#include "knn.cuh"
#include "odom.cuh"
#include "qr.cuh"
#include "solver_dev.cuh"
#include "solver_host.h"
#include "voxel.cuh"
#include <chrono>
#include <cstddef>
#include <memory>
#include <new>
#include <vector>

namespace lio {
using namespace hm;

constexpr int kMaxWindow = 32;

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// ------------------------------------------------------------------------------------------------
// kernels
struct ConcatParams {
  const float4 *src[kMaxWindow];
  const int *n[kMaxWindow];
  float R[kMaxWindow][9];
  float t[kMaxWindow][3];
  float tag[kMaxWindow];
  int identity[kMaxWindow];  // copy as is (pivot frame keeps its intensity)
  int skip_first[kMaxWindow];  // drop the first k points (SlideWindow ExtractIndices), value read from *skip_n
  const int *skip_n[kMaxWindow];
  int nsrc;
};

// pcl::transformPointCloud (x' = m00 x + m01 y + m02 z + m03, left to right) + intensity tag + concat
// (Estimator.cc:1498-1507, :2600-2611).  Exact float order: compiled with -fmad=false.
__global__ void __launch_bounds__(256)
k_concat(const ConcatParams P, float4 *__restrict__ dst, int *__restrict__ n_out, int cap) {
  __shared__ int off[kMaxWindow + 1];
  __shared__ int skip[kMaxWindow];
  if (threadIdx.x == 0) {
    int run = 0;
    for (int k = 0; k < P.nsrc; ++k) {
      int sk = P.skip_first[k] ? *P.skip_n[k] : 0;
      int nk = *P.n[k] - sk;
      if (nk < 0) nk = 0;
      skip[k] = sk;
      off[k] = run;
      run += nk;
    }
    off[P.nsrc] = run;
    if (blockIdx.x == 0) *n_out = run < cap ? run : cap;
  }
  __syncthreads();
  const int total = min(off[P.nsrc], cap);
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
    int k = 0;
    while (k + 1 < P.nsrc && g >= off[k + 1]) ++k;
    float4 p = __ldg(P.src[k] + (g - off[k]) + skip[k]);
    if (!P.identity[k]) {
      const float *R = P.R[k];
      const float *t = P.t[k];
      float x = R[0] * p.x + R[1] * p.y + R[2] * p.z + t[0];
      float y = R[3] * p.x + R[4] * p.y + R[5] * p.z + t[1];
      float z = R[6] * p.x + R[7] * p.y + R[8] * p.z + t[2];
      p = make_float4(x, y, z, P.tag[k] >= 0.f ? P.tag[k] : p.w);
    }
    dst[g] = p;
  }
}

__device__ __forceinline__ void qmul_vec(float qx, float qy, float qz, float qw, float vx, float vy, float vz, float &ox, float &oy, float &oz) {
  float ux = qy * vz - qz * vy, uy = qz * vx - qx * vz, uz = qx * vy - qy * vx;
  ux += ux; uy += uy; uz += uz;
  float cx = qy * uz - qz * uy, cy = qz * ux - qx * uz, cz = qx * uy - qy * ux;
  ox = vx + ux * qw + cx; oy = vy + uy * qw + cy; oz = vz + uz * qw + cz;
}

// TransformToEnd (Estimator.cc:62-103), in place
__global__ void __launch_bounds__(256)
k_deskew(float4 *__restrict__ cloud, const int *__restrict__ n_dev, TransformF es, float time_factor) {
  const int n = *n_dev;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = cloud[i];
  float s = time_factor * (p.w - (float)(int)p.w);
  p.x -= s * es.px; p.y -= s * es.py; p.z -= s * es.pz;
  p.w -= (float)(int)p.w;
  // q_s = identity.slerp(s, q_e)  (Eigen QuaternionBase::slerp)
  const float one = 1.0f - FLT_EPSILON;
  float d = es.qw;  // identity . q_e
  float absD = fabsf(d);
  float scale0, scale1;
  if (absD >= one) { scale0 = 1.0f - s; scale1 = s; }
  else {
    float theta = acosf(absD);
    float sinTheta = sinf(theta);
    scale0 = sinf((1.0f - s) * theta) / sinTheta;
    scale1 = sinf(s * theta) / sinTheta;
  }
  if (d < 0.f) scale1 = -scale1;
  float sw = scale0 + scale1 * es.qw, sx = scale1 * es.qx, sy = scale1 * es.qy, sz = scale1 * es.qz;
  // q_s.conjugate().normalized()
  float nn = sqrtf(sx * sx + sy * sy + sz * sz + sw * sw);
  float cx = -sx / nn, cy = -sy / nn, cz = -sz / nn, cw = sw / nn;
  float ax, ay, az;
  qmul_vec(cx, cy, cz, cw, p.x, p.y, p.z, ax, ay, az);
  float bx, by, bz;
  qmul_vec(es.qx, es.qy, es.qz, es.qw, ax, ay, az, bx, by, bz);
  cloud[i] = make_float4(bx + es.px, by + es.py, bz + es.pz, p.w);
}

constexpr int kOdomThreads = 256;

__global__ void __launch_bounds__(kOdomThreads)
k_odom_reduce(const float4 *__restrict__ pts, const float4 *__restrict__ coef, const int *__restrict__ n_dev,
              const TransformF *__restrict__ tf_dev, OdomState *__restrict__ st, double *__restrict__ partial, int mode = 0) {
  __shared__ double sred[kOdomThreads / 32][27];
  __shared__ bool is_last;
  if (st->done) return;
  const int n = *n_dev;
  const TransformF tf = *tf_dev;
  // rot.toRotationMatrix() of the (possibly un-normalised) quaternion, float
  float R[9];
  {
    const float tx = 2.f * tf.qx, ty = 2.f * tf.qy, tz = 2.f * tf.qz;
    const float twx = tx * tf.qw, twy = ty * tf.qw, twz = tz * tf.qw, txx = tx * tf.qx, txy = ty * tf.qx, txz = tz * tf.qx;
    const float tyy = ty * tf.qy, tyz = tz * tf.qy, tzz = tz * tf.qz;
    R[0] = 1.f - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
    R[3] = txy + twz; R[4] = 1.f - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1.f - (txx + tyy);
  }
  // mode 2 (MapBuilder::OptimizeMap, MapBuilder.cc:905-911): J_r is post-multiplied by rot.inverse().toRotationMatrix()
  // (inverse = conjugate / squaredNorm) and the rotation information matrix diag(5e-3, 5e-3, 1)
  float Ri[9];
  {
    const float n2 = tf.qx * tf.qx + tf.qy * tf.qy + tf.qz * tf.qz + tf.qw * tf.qw;
    const float ix = -tf.qx / n2, iy = -tf.qy / n2, iz = -tf.qz / n2, iw = tf.qw / n2;
    const float tx = 2.f * ix, ty = 2.f * iy, tz = 2.f * iz;
    const float twx = tx * iw, twy = ty * iw, twz = tz * iw, txx = tx * ix, txy = ty * ix, txz = tz * ix;
    const float tyy = ty * iy, tyz = tz * iy, tzz = tz * iz;
    Ri[0] = 1.f - (tyy + tzz); Ri[1] = txy - twz; Ri[2] = txz + twy;
    Ri[3] = txy + twz; Ri[4] = 1.f - (txx + tzz); Ri[5] = tyz - twx;
    Ri[6] = txz - twy; Ri[7] = tyz + twx; Ri[8] = 1.f - (txx + tyy);
  }
  double acc[27];
#pragma unroll
  for (int k = 0; k < 27; ++k) acc[k] = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = __ldg(pts + i), c = __ldg(coef + i);
    // RS = R * skew(p);  J_r = -w^T RS,  J_t = w^T
    float RS[9];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      RS[r * 3 + 0] = R[r * 3 + 1] * p.z + R[r * 3 + 2] * (-p.y);
      RS[r * 3 + 1] = R[r * 3 + 0] * (-p.z) + R[r * 3 + 2] * p.x;
      RS[r * 3 + 2] = R[r * 3 + 0] * p.y + R[r * 3 + 1] * (-p.x);
    }
    float row[6];
#pragma unroll
    for (int q = 0; q < 3; ++q) row[q] = -(c.x * RS[q] + c.y * RS[3 + q] + c.z * RS[6 + q]);
    if (mode == 2) {
      const float t0 = row[0] * Ri[0] + row[1] * Ri[3] + row[2] * Ri[6];
      const float t1 = row[0] * Ri[1] + row[1] * Ri[4] + row[2] * Ri[7];
      const float t2 = row[0] * Ri[2] + row[1] * Ri[5] + row[2] * Ri[8];
      row[0] = t0 * 5e-3f; row[1] = t1 * 5e-3f; row[2] = t2 * 1.0f;
    }
    row[3] = c.x; row[4] = c.y; row[5] = c.z;
    float rx, ry, rz;
    qmul_vec(tf.qx, tf.qy, tf.qz, tf.qw, p.x, p.y, p.z, rx, ry, rz);
    // CalculateLaserOdom: d2 = w . (R p + t) + b (Estimator.cc:1282-1284); scan-to-map: d2 = coeff.intensity (PointMapping.cc:634)
    float d2 = mode != 0 ? c.w : c.x * (rx + tf.px) + c.y * (ry + tf.py) + c.z * (rz + tf.pz) + c.w;
    int k = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
#pragma unroll
      for (int b = a; b < 6; ++b) acc[k++] += (double)(row[a] * row[b]);
    }
#pragma unroll
    for (int a = 0; a < 6; ++a) acc[21 + a] += (double)(row[a] * (-d2));
  }
#pragma unroll
  for (int k = 0; k < 27; ++k) {
    double v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane_id() == 0) sred[warp_id()][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 27) {
    double v = 0;
#pragma unroll
    for (int w = 0; w < kOdomThreads / 32; ++w) v += sred[w][threadIdx.x];
    partial[blockIdx.x * 32 + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(&st->counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (threadIdx.x < 27) {
    double v = 0;
    for (unsigned b = 0; b < gridDim.x; ++b) v += __ldcg(partial + b * 32 + threadIdx.x);
    if (threadIdx.x < 21) {
      int k = threadIdx.x, a = 0;
      while (k >= 6 - a) { k -= 6 - a; ++a; }
      int b = a + k;
      st->AtA[a * 6 + b] = v; st->AtA[b * 6 + a] = v;
    } else {
      st->AtB[threadIdx.x - 21] = v;
    }
  }
  if (threadIdx.x == 0) st->counter = 0u;
}

__global__ void k_odom_solve(OdomState *__restrict__ st, TransformF *__restrict__ tf_dev, double delta_r_abort, double delta_t_abort,
                             int round = -1, const int *__restrict__ n_dev = nullptr, int min_features = 0, int left_update = 0) {
  if (threadIdx.x != 0 || st->done) return;
  odom_solve_step(st, tf_dev, delta_r_abort, delta_t_abort, round, n_dev, min_features, left_update);
}

// One CalculateLaserOdom round after the k-NN launch, as a single CTA: reduce the round's features (float products
// accumulated in double, fixed thread -> feature mapping and a fixed reduction tree: deterministic), solve, and zero the
// k-NN launch state (tile status words, ticket) so that the next round's k-NN launch needs no memset.
constexpr int kOdomRoundThreads = 512;
__global__ void __launch_bounds__(kOdomRoundThreads)
k_odom_round(const float4 *__restrict__ pts, const float4 *__restrict__ coef, const int *__restrict__ n_dev, TransformF *__restrict__ tf_dev,
             OdomState *__restrict__ st, double delta_r_abort, double delta_t_abort, unsigned long long *__restrict__ knn_status, int knn_ntiles,
             int *__restrict__ knn_ticket) {
  __shared__ double sred[kOdomRoundThreads / 32][27];
  if (st->done) return;   // the k-NN launch of a finished chain was a no-op: nothing to clean
  const int n = *n_dev;
  const TransformF tf = *tf_dev;
  float R[9];
  odom_rotation(tf, R);
  double acc[27];
#pragma unroll
  for (int k = 0; k < 27; ++k) acc[k] = 0.0;
  // four features per trip: their eight loads are issued together (the loop is latency bound: ~25 features per thread)
#pragma unroll 1
  for (int i0 = threadIdx.x; i0 < n; i0 += 4 * kOdomRoundThreads) {
    float4 pq[4], cq[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * kOdomRoundThreads;
      if (i < n) { pq[u] = __ldg(pts + i); cq[u] = __ldg(coef + i); }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
    if (i0 + u * kOdomRoundThreads >= n) break;
    float row[6], d2;
    odom_row(tf, R, pq[u], cq[u], row, d2);
    int k = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
#pragma unroll
      for (int b = a; b < 6; ++b) acc[k++] += (double)(row[a] * row[b]);
    }
#pragma unroll
    for (int a = 0; a < 6; ++a) acc[21 + a] += (double)(row[a] * (-d2));
    }
  }
#pragma unroll
  for (int k = 0; k < 27; ++k) {
    double v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane_id() == 0) sred[warp_id()][k] = v;
  }
  for (int t = threadIdx.x; t < knn_ntiles; t += kOdomRoundThreads) knn_status[t] = 0ull;
  if (threadIdx.x == 0) *knn_ticket = 0;
  __syncthreads();
  if (threadIdx.x < 27) {
    double v = 0;
#pragma unroll
    for (int w = 0; w < kOdomRoundThreads / 32; ++w) v += sred[w][threadIdx.x];
    if (threadIdx.x < 21) {
      int k = threadIdx.x, a = 0;
      while (k >= 6 - a) { k -= 6 - a; ++a; }
      const int b = a + k;
      st->AtA[a * 6 + b] = v; st->AtA[b * 6 + a] = v;
    } else {
      st->AtB[threadIdx.x - 21] = v;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) odom_solve_step(st, tf_dev, delta_r_abort, delta_t_abort);
}

}  // namespace lio

// ------------------------------------------------------------------------------------------------
using namespace lio;
using namespace lio::hm;

struct lio_pim {
  std::shared_ptr<Preintegration> p;
};

struct ImuStampedF {
  double time;
  float q[4];  // x y z w
  float p[3];
};

struct MargPrior {
  bool valid = false;
  int n = 0;      // 15*O + 6
  Mat Hp;         // J^T J
  Vec bp;         // J^T r0
  double c0 = 0;  // r0^T r0
  std::vector<double> x0_pose, x0_sb;  // O x 7, O x 9
  double x0_ex[7];
};

// Marginalisation split in two: the linearised system (A, b) of the dropped + kept blocks is built right after the
// solve (it needs the device reduction and the converged parameters); the dense algebra (Schur complement + two
// symmetric eigen-decompositions, ~n^3) is a pure function of that snapshot and runs on a worker thread while the next
// scan's front end (deskew, voxel grid, local map, k-NN features) keeps the device busy.  The worker is started at
// the ENTRY of the next lio_est_process_scan_* call, not earlier, so none of it runs outside a caller's timed step.
constexpr size_t kXRowBytes = sizeof(double) * kMaxOpt * kAsmStride;
constexpr size_t kXFlagOff = 2 * kXRowBytes;
constexpr size_t kXErrOff = kXFlagOff + sizeof(unsigned) * kMaxPeers;
constexpr size_t kXBytes = kXErrOff + 64;

struct MargJob {
  bool stashed = false, running = false;
  int O = 0;
  Mat A;
  Vec b;
  std::vector<double> x0_pose, x0_sb;
  double x0_ex[7];
  MargPrior result;
};

// One persistent helper thread per estimator context (created on first use): starting a std::thread per scan costs
// ~0.1 ms on the bench host.  Hand-off: the helper spins for spin_us after each job before it sleeps on the condition
// variable, so the jobs of one solve (one every ~150 us) never pay a futex wake-up; between scans it sleeps.
struct Worker {
  double spin_us = 400.0;   // hand-off spin window; shortened for sharded runs (one process per GPU shares the host cores)
  std::thread th;
  std::mutex mu;
  std::condition_variable cv;
  std::function<void()> job;
  std::atomic<int> has_job{0}, busy{0}, sleeping{0};
  bool quit = false, started = false;
  static inline void relax() {
#if defined(__x86_64__)
    __builtin_ia32_pause();
#endif
  }
  void submit(std::function<void()> f) {
    wait();                                // the previous job has fully retired
    if (!started) { started = true; th = std::thread([this]() { loop(); }); }
    job = std::move(f);
    busy.store(1);
    has_job.store(1);
    if (sleeping.load()) { std::lock_guard<std::mutex> lk(mu); cv.notify_all(); }
  }
  void wait() {
    const double t0 = now_s();
    while (busy.load()) {
      relax();
      if ((now_s() - t0) * 1e6 > spin_us) {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [this]() { return busy.load() == 0; });
        return;
      }
    }
  }
  void loop() {
    while (true) {
      const double t0 = now_s();
      bool got = false;
      while ((now_s() - t0) * 1e6 <= spin_us) {
        if (has_job.load()) { got = true; break; }
        relax();
      }
      if (!got) {
        std::unique_lock<std::mutex> lk(mu);
        sleeping.store(1);
        cv.wait(lk, [this]() { return has_job.load() != 0 || quit; });
        sleeping.store(0);
        if (!has_job.load()) return;  // quit
      }
      has_job.store(0);
      job();
      busy.store(0);
      { std::lock_guard<std::mutex> lk(mu); cv.notify_all(); }
    }
  }
  ~Worker() {
    if (started) {
      wait();
      { std::lock_guard<std::mutex> lk(mu); quit = true; cv.notify_all(); }
      th.join();
    }
  }
};

struct lio_est {
  lio_est_config cfg;
  MargJob mjob;
  Worker worker;
  // fused exchange over peer memory (multi-GPU): one device allocation per rank, laid out as
  //   [2 parities][kMaxOpt * kAsmStride doubles] | unsigned flag[kMaxPeers] | int err
  char *xbuf = nullptr;
  char *peer_base[kMaxPeers] = {};
  int npeers = 0;
  unsigned xepoch = 0;
  Mat hp_exp;              // prior Hp scattered into the current tangent layout (cache of one solve)
  bool hp_exp_valid = false;
  struct ImuBlockStore { double JtJ[30 * 30], Jtr[30], cost; bool used; } imu_blocks_store[kMaxOpt];
  std::atomic<int> imu_next{0}, imu_done{0};  // shared pool of ImuFactor indices of one linearisation (caller + helper)
  double t_marg_wait = 0;
  char err[512] = "";         // text of the last failed call on THIS handle (lio_est_last_error)
  bool window_open = false;   // between lio_est_open_scan_* and lio_est_close_scan (stepwise API)
  bool poisoned = false;   // a scan failed half-way: the window bookkeeping is inconsistent, every later call fails fast
  int W = 0, O = 0, device = 0;
  cudaStream_t stream = 0;
  int sm_count = 148;
  // ---- host window state
  std::vector<V3> Ps, Vs, Bas, Bgs;
  std::vector<M3> Rs;
  std::vector<std::shared_ptr<Preintegration>> pre;
  std::shared_ptr<Preintegration> tmp_pre;
  ImuNoise noise;
  V3 acc_last, gyr_last, g_vec;
  bool first_imu = false;
  float tlb_q[4] = {0, 0, 0, 1}, tlb_p[3] = {0, 0, -0.1f};  // transform_lb_ (Twist<float>)
  std::vector<ImuStampedF> imu_stamped;
  std::vector<std::vector<double>> para_pose, para_sb;
  double para_ex[7];
  MargPrior prior;
  bool convergence_flag = false, init_local_map = false;
  int extrinsic_stage = 1;
  bool ex_constant = false;
  // ---- device
  std::vector<float4 *> slot_ptr;    // physical slots
  std::vector<int> slot_of;          // logical frame -> physical slot
  int *d_slot_n = nullptr;           // counts per physical slot
  std::vector<int> size_surf_stack;  // host mirror of each frame's own size (logical)
  int *d_own_n = nullptr;            // device: own size per physical slot (for SlideWindow's skip)
  int slot_cap = 0;
  float4 *d_scan = nullptr, *d_local = nullptr, *d_map = nullptr, *d_tmp = nullptr;
  int local_cap = 0;
  int *d_counts = nullptr;  // [0] scan n [1] local n [2] map n [3] tmp n
  VoxelGrid vg;
  CellHash hash;
  KnnWork knn;
  KnnWork knn2;                     // launch state of the LaserOdom chain, which runs beside the frame-batched k-NN launch
  cudaStream_t ostream = nullptr;   // stream of that chain
  cudaEvent_t ev_map = nullptr, ev_odom = nullptr;
  std::vector<FeatureOut> feats;  // logical frame index
  int *d_feat_counts = nullptr;   // W+1 (inside the feature slab, current parity)
  // All feature buffers (xyz+score, coefficients, counts) live in ONE allocation with two parities, so that a sharded run can
  // exchange the features themselves once per scan (lio_est_set_feature_peers): every rank then owns all frames' features and the
  // whole solve runs exactly like a single-GPU solve - no rendezvous inside the 11 evaluations.
  char *fslab = nullptr;
  size_t fslab_bytes = 0, fpar_stride = 0, foff_cnt = 0, foff_flags = 0;
  std::vector<size_t> foff_pts, foff_coef;
  bool fpeers = false;
  char *fpeer_base[kMaxPeers] = {};
  unsigned fepoch = 0;
  int fparity = 0;
  TransformF *d_tf = nullptr;     // W+1
  TransformF *h_tf = nullptr;     // pinned
  AsmWork asmw;
  double *h_Rt = nullptr;   // pinned kMaxOpt*kAsmRtStride
  double *d_Rt = nullptr;
  double *h_S = nullptr;    // pinned kMaxOpt*kAsmStride
  int *h_counts = nullptr;  // pinned
  OdomState *d_odom = nullptr;
  double *d_odom_partial = nullptr;
  // ---- sharding
  int rank = 0, world = 1;
  lio_allreduce_fn allreduce = nullptr;
  void *allreduce_user = nullptr;
  // ---- results / stats
  std::vector<int> h_feat_n;
  int h_map_n = 0;
  std::vector<TransformF> local_tf;
  DoglegSummary summary;
  double cost_pim = 0, cost_ppp = 0, cost_marg = 0;
  bool turn_off = true;
  int odom_iters = 0;
  double t_build = 0, t_feat = 0, t_solve = 0, t_marg = 0, t_total = 0;
  bool S_pending = false;
  long long S_pending_feats = 0;
  double t_lin_wait = 0, t_lin_host = 0, t_lin_lidar = 0;  // per scan: blocked on the device / host factor work / lidar block expansion
  int launches = 0;
  Mat H0;
  Vec g0;
  double cost0 = 0;
  bool have_H0 = false;
  // device-resident solver
  DevSolver ds;
  bool use_dev_solver = false;
  // the device solver's launches of one solve, captured once and replayed (single-GPU contexts)
  cudaStream_t gstream = nullptr;
  cudaGraph_t sgraph = nullptr;
  cudaGraphExec_t sexec = nullptr;
  std::vector<cudaGraphNode_t> asm_nodes;
  cudaEvent_t ev_gin = nullptr, ev_gout = nullptr;
  int graph_launches = 0;
  bool prior_uploaded = false;
  bool ds_prepared = false, ds_prepared_asm = false;   // solve_dev_prepare ran for the current parameters
  int ds_prepared_it = 0;
  cudaEvent_t evp[2 * 24] = {};
  // cached lidar reduction for the current parameter values
  bool S_valid = false;
  // CUDA-event timing of the fused kernel (on the launching stream)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr;
  double knn_ms_sum = 0;
  long long knn_launch_count = 0, knn_query_sum = 0;
  bool knn_timed = false;
  double asm_ms_sum = 0;
  long long asm_launch_count = 0, asm_feat_sum = 0;
};

static Tw tlb_double(const lio_est *e) {
  return Tw(Q(e->tlb_q[3], e->tlb_q[0], e->tlb_q[1], e->tlb_q[2]), V3(e->tlb_p[0], e->tlb_p[1], e->tlb_p[2]));
}

static Tw lidar_pose(const V3 &P, const M3 &R, const Tw &tlb) {  // Estimator.cc:1387-1390
  Q rot = fromR(R * toR(inverse(tlb.rot)));
  V3 pos = P - rotate(rot, tlb.pos);
  return Tw(rot, pos);
}

// Twist<double> -> cast<float>() -> transform(): float quaternion normalised in float, float matrix
struct AffineF { float R[9]; float t[3]; TransformF tf; };
static AffineF to_affine_f(const Tw &t) {
  AffineF a;
  float qx = (float)t.rot.x, qy = (float)t.rot.y, qz = (float)t.rot.z, qw = (float)t.rot.w;
  float n = std::sqrt(qx * qx + qy * qy + qz * qz + qw * qw);
  qx /= n; qy /= n; qz /= n; qw /= n;
  const float tx = 2.f * qx, ty = 2.f * qy, tz = 2.f * qz;
  const float twx = tx * qw, twy = ty * qw, twz = tz * qw, txx = tx * qx, txy = ty * qx, txz = tz * qx;
  const float tyy = ty * qy, tyz = tz * qy, tzz = tz * qz;
  a.R[0] = 1.f - (tyy + tzz); a.R[1] = txy - twz; a.R[2] = txz + twy;
  a.R[3] = txy + twz; a.R[4] = 1.f - (txx + tzz); a.R[5] = tyz - twx;
  a.R[6] = txz - twy; a.R[7] = tyz + twx; a.R[8] = 1.f - (txx + tyy);
  a.t[0] = (float)t.pos.x; a.t[1] = (float)t.pos.y; a.t[2] = (float)t.pos.z;
  // Twist<float>(Affine3f): Quaternionf(linear).normalized()
  float m[3][3] = {{a.R[0], a.R[1], a.R[2]}, {a.R[3], a.R[4], a.R[5]}, {a.R[6], a.R[7], a.R[8]}};
  float q[4];
  float tr = m[0][0] + m[1][1] + m[2][2];
  if (tr > 0.f) {
    float s = std::sqrt(tr + 1.0f);
    q[3] = 0.5f * s;
    s = 0.5f / s;
    q[0] = (m[2][1] - m[1][2]) * s; q[1] = (m[0][2] - m[2][0]) * s; q[2] = (m[1][0] - m[0][1]) * s;
  } else {
    int i = 0;
    if (m[1][1] > m[0][0]) i = 1;
    if (m[2][2] > m[i][i]) i = 2;
    int j = (i + 1) % 3, k = (j + 1) % 3;
    float s = std::sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0f);
    q[i] = 0.5f * s;
    s = 0.5f / s;
    q[3] = (m[k][j] - m[j][k]) * s;
    q[j] = (m[j][i] + m[i][j]) * s;
    q[k] = (m[k][i] + m[i][k]) * s;
  }
  float qn = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  a.tf.qx = q[0] / qn; a.tf.qy = q[1] / qn; a.tf.qz = q[2] / qn; a.tf.qw = q[3] / qn;
  a.tf.px = a.t[0]; a.tf.py = a.t[1]; a.tf.pz = a.t[2];
  return a;
}

template <typename T> static void push_shift(std::vector<T> &v, T x) { v.erase(v.begin()); v.push_back(x); }

#define EST_CUDA(expr) LIO_CUDA_OK(expr)

// ---- creation -----------------------------------------------------------------------------------
extern "C" void lio_est_default_config(lio_est_config *c) {
  c->window_size = 10; c->opt_window_size = 10;
  c->min_match_sq_dis = 1.0f; c->min_plane_dis = 0.2f; c->surf_filter_size = 0.4f;
  c->keep_features = 0; c->estimate_extrinsic = 1; c->opt_extrinsic = 1;
  c->imu_factor = 1; c->point_distance_factor = 1; c->prior_factor = 0; c->marginalization_factor = 1;
  c->enable_deskew = 1; c->cutoff_deskew = 1;
  c->acc_n = 0.2; c->gyr_n = 0.02; c->acc_w = 2e-4; c->gyr_w = 2e-5; c->g_norm = 9.805;
  c->max_num_iterations = 10; c->odom_max_iterations = 10;
  c->max_frame_points = 1 << 16; c->max_scan_points = 1 << 18;
  c->device_solver = 1;   // GPU-resident dogleg loop (solver_dev.cu); 0 keeps the host controller (also used when O > 13)
  c->overlap_marginalization = 1;
  c->solver_graph = 1;
}

// point the per-frame feature descriptors at one parity of the slab
static void set_feature_parity(lio_est *e, int par) {
  char *base = e->fslab + (size_t)par * e->fpar_stride;
  e->d_feat_counts = reinterpret_cast<int *>(base + e->foff_cnt);
  const int pivot = e->W - e->O;
  for (int k = pivot + 1; k <= e->W; ++k) {
    FeatureOut &f = e->feats[k];
    f.pts = reinterpret_cast<float4 *>(base + e->foff_pts[k]);
    f.coef = reinterpret_cast<float4 *>(base + e->foff_coef[k]);
    f.count = e->d_feat_counts + k;
  }
  e->fparity = par;
}

// ---- per-scan feature exchange over peer memory (sharded runs) ----------------------------------------------------------
struct FeaturePeers {
  float4 *pts[kMaxPeers], *coef[kMaxPeers];
  int *count[kMaxPeers];
  int npeers, self;
};
// An owned frame's features go to the same place in every peer's slab (plain P2P stores over NVLink / NVSwitch).
__global__ void __launch_bounds__(256)
k_publish_features(const float4 *__restrict__ pts, const float4 *__restrict__ coef, const int *__restrict__ count, int cap, FeaturePeers P) {
  const int n = min(*count, cap);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 v = pts[i], w = coef[i];
    for (int r = 0; r < P.npeers; ++r) if (r != P.self) { P.pts[r][i] = v; P.coef[r][i] = w; }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) for (int r = 0; r < P.npeers; ++r) if (r != P.self) *P.count[r] = *count;
}
struct FlagPeers { unsigned *flag[kMaxPeers]; int npeers, self; };
// after the publishing kernels of this rank have completed (stream order): the scan's epoch into every rank's flag slot
__global__ void k_publish_flag(FlagPeers P, unsigned epoch) {
  __threadfence_system();
  if ((int)threadIdx.x < P.npeers) {
    unsigned *fl = P.flag[threadIdx.x] + P.self;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(fl), "r"(epoch) : "memory");
  }
}

extern "C" int lio_est_destroy(lio_est *e) {
  if (!e) return LIO_OK;
  if (e->mjob.running) { e->worker.wait(); e->mjob.running = false; }
  cudaSetDevice(e->device);
  for (float4 *p : e->slot_ptr) if (p) cudaFree(p);
  for (FeatureOut &f : e->feats) if (f.src) cudaFree(f.src);
  void *ptrs[] = {e->d_slot_n, e->d_own_n, e->d_scan, e->d_local, e->d_map, e->d_tmp, e->d_counts, e->fslab, e->d_tf, e->d_odom, e->d_odom_partial};
  for (void *p : ptrs) if (p) cudaFree(p);
  for (int k = 0; k < 48; ++k) if (e->evp[k]) cudaEventDestroy(e->evp[k]);
  e->ds.destroy();
  if (e->sexec) cudaGraphExecDestroy(e->sexec);
  if (e->sgraph) cudaGraphDestroy(e->sgraph);
  if (e->gstream) cudaStreamDestroy(e->gstream);
  if (e->ev_gin) cudaEventDestroy(e->ev_gin);
  if (e->ev_gout) cudaEventDestroy(e->ev_gout);
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  if (e->evk0) cudaEventDestroy(e->evk0);
  if (e->evk1) cudaEventDestroy(e->evk1);
  if (e->xbuf) cudaFree(e->xbuf);
  if (e->h_tf) cudaFreeHost(e->h_tf);
  if (e->h_S) cudaFreeHost(e->h_S);
  if (e->h_Rt) cudaFreeHost(e->h_Rt);
  if (e->d_Rt) cudaFree(e->d_Rt);
  if (e->h_counts) cudaFreeHost(e->h_counts);
  e->vg.destroy(); e->hash.destroy(); e->knn.destroy(); e->knn2.destroy(); e->asmw.destroy();
  if (e->ostream) cudaStreamDestroy(e->ostream);
  if (e->ev_map) cudaEventDestroy(e->ev_map);
  if (e->ev_odom) cudaEventDestroy(e->ev_odom);
  delete e;
  return LIO_OK;
}

extern "C" int lio_est_create(const lio_est_config *cfg, int device, void *cuda_stream, lio_est **out) {
  if (!cfg || !out) return LIO_ERR_INVALID;
  const int W = cfg->window_size, O = cfg->opt_window_size;
  if (W < 1 || W >= kMaxWindow || O < 1 || O > W || O > kMaxOpt || cfg->max_frame_points < 16 || cfg->max_scan_points < 16 ||
      !(cfg->surf_filter_size > 0) || !(cfg->min_match_sq_dis > 0) || cfg->odom_max_iterations < 1) {
    lio_set_last_error(__FILE__, __LINE__, "lio_est_create: configuration outside supported limits");
    return LIO_ERR_INVALID;
  }
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  LIO_CUDA_OK(cudaSetDevice(device));
  lio_est *e = new (std::nothrow) lio_est();
  if (!e) return LIO_ERR_INVALID;
  e->cfg = *cfg; e->W = W; e->O = O; e->device = device; e->stream = (cudaStream_t)cuda_stream;
  cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, device);
  e->noise.acc_n = cfg->acc_n; e->noise.gyr_n = cfg->gyr_n; e->noise.acc_w = cfg->acc_w; e->noise.gyr_w = cfg->gyr_w; e->noise.g_norm = cfg->g_norm;
  e->g_vec = V3(0, 0, -cfg->g_norm);
  e->extrinsic_stage = cfg->estimate_extrinsic;
  e->Ps.assign(W + 1, V3()); e->Vs.assign(W + 1, V3()); e->Bas.assign(W + 1, V3()); e->Bgs.assign(W + 1, V3());
  e->Rs.assign(W + 1, M3::I());
  e->pre.assign(W + 1, nullptr);
  e->para_pose.assign(O + 1, std::vector<double>(7, 0.0));
  e->para_sb.assign(O + 1, std::vector<double>(9, 0.0));
  std::memset(e->para_ex, 0, sizeof(e->para_ex));
  e->size_surf_stack.assign(W + 1, 0);
  e->h_feat_n.assign(W + 1, 0);
  e->local_tf.assign(W + 1, TransformF{0, 0, 0, 1, 0, 0, 0});
  const int pivot = W - O;
  e->slot_cap = cfg->max_frame_points * (pivot + 1);
  e->slot_ptr.assign(W + 1, nullptr);
  e->slot_of.resize(W + 1);
  bool ok = true;
  for (int k = 0; k <= W; ++k) {
    e->slot_of[k] = k;
    ok = ok && cudaMalloc(&e->slot_ptr[k], sizeof(float4) * e->slot_cap) == cudaSuccess;
  }
  e->local_cap = e->slot_cap + cfg->max_frame_points * (O > 1 ? O - 1 : 1);
  ok = ok && cudaMalloc(&e->d_slot_n, sizeof(int) * (W + 1)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_own_n, sizeof(int) * (W + 1)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_scan, sizeof(float4) * cfg->max_scan_points) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_local, sizeof(float4) * e->local_cap) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_map, sizeof(float4) * e->local_cap) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_tmp, sizeof(float4) * e->slot_cap) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_counts, sizeof(int) * 8) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_tf, sizeof(TransformF) * (W + 1)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_odom, sizeof(OdomState)) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_odom_partial, sizeof(double) * 32 * 1024) == cudaSuccess;
  ok = ok && cudaMallocHost((void **)&e->h_tf, sizeof(TransformF) * (W + 1)) == cudaSuccess;
  ok = ok && cudaMallocHost((void **)&e->h_S, sizeof(double) * (kMaxOpt * kAsmStride + 2)) == cudaSuccess;  // + exchange error flag
  if (ok) std::memset(e->h_S, 0, sizeof(double) * (kMaxOpt * kAsmStride + 2));
  ok = ok && cudaMallocHost((void **)&e->h_Rt, sizeof(double) * kMaxOpt * kAsmRtStride) == cudaSuccess;
  ok = ok && cudaMalloc(&e->d_Rt, sizeof(double) * kMaxOpt * kAsmRtStride) == cudaSuccess;
  ok = ok && cudaMallocHost((void **)&e->h_counts, sizeof(int) * (W + 16)) == cudaSuccess;
  int vg_cap = std::max(e->local_cap, cfg->max_scan_points);
  ok = ok && e->vg.init(vg_cap) == 0;
  ok = ok && e->hash.init(e->local_cap) == 0;
  ok = ok && e->knn.init(cfg->max_frame_points * (O + 1)) == 0;
  ok = ok && e->knn2.init(cfg->max_frame_points) == 0;
  ok = ok && cudaStreamCreateWithFlags(&e->ostream, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&e->ev_map, cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&e->ev_odom, cudaEventDisableTiming) == cudaSuccess;
  e->feats.assign(W + 1, FeatureOut());
  long long total_feat = 0;
  {
    e->foff_pts.assign(W + 1, 0); e->foff_coef.assign(W + 1, 0);
    size_t off = 0;
    for (int k = pivot + 1; k <= W; ++k) {
      const int cap = cfg->max_frame_points * ((k == W && cfg->keep_features) ? cfg->odom_max_iterations : 1);
      e->feats[k].cap = cap;
      e->foff_pts[k] = off; off += sizeof(float4) * (size_t)cap;
      e->foff_coef[k] = off; off += sizeof(float4) * (size_t)cap;
      total_feat += cap;
    }
    e->foff_cnt = off; off += ((sizeof(int) * (size_t)(W + 1) + 255) / 256) * 256;
    e->fpar_stride = off;
    e->foff_flags = 2 * off;
    e->fslab_bytes = 2 * off + 256;   // epoch flags (one per source rank) + error word behind the two parities
    ok = ok && cudaMalloc(&e->fslab, e->fslab_bytes) == cudaSuccess && cudaMemset(e->fslab, 0, e->fslab_bytes) == cudaSuccess;
    for (int k = pivot + 1; k <= W && ok; ++k) ok = ok && cudaMalloc(&e->feats[k].src, sizeof(int) * e->feats[k].cap) == cudaSuccess;
    if (ok) set_feature_parity(e, 0);
  }
  ok = ok && e->asmw.init((int)std::min<long long>(total_feat, 1ll << 30)) == 0;
  if (ok) {
    ok = ok && cudaMemset(e->d_slot_n, 0, sizeof(int) * (W + 1)) == cudaSuccess;
    ok = ok && cudaMemset(e->d_own_n, 0, sizeof(int) * (W + 1)) == cudaSuccess;
    ok = ok && cudaMemset(e->d_counts, 0, sizeof(int) * 8) == cudaSuccess;
  }
  ok = ok && cudaEventCreate(&e->ev0) == cudaSuccess && cudaEventCreate(&e->ev1) == cudaSuccess;
  ok = ok && cudaEventCreate(&e->evk0) == cudaSuccess && cudaEventCreate(&e->evk1) == cudaSuccess;
  ok = ok && cudaMalloc(&e->xbuf, kXBytes) == cudaSuccess && cudaMemset(e->xbuf, 0, kXBytes) == cudaSuccess;
  for (int k = 0; k < 48 && ok; ++k) ok = ok && cudaEventCreate(&e->evp[k]) == cudaSuccess;
  e->use_dev_solver = cfg->device_solver != 0 && e->ds.supports(O) && cfg->max_num_iterations <= 22;
  if (e->use_dev_solver) ok = ok && e->ds.init(O) == 0;
  if (e->use_dev_solver && cfg->solver_graph) {
    ok = ok && cudaStreamCreateWithFlags(&e->gstream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&e->ev_gin, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&e->ev_gout, cudaEventDisableTiming) == cudaSuccess;
  }
  if (!ok) {
    lio_set_last_error(__FILE__, __LINE__, "lio_est_create: device allocation failed");
    lio_est_destroy(e);
    return LIO_ERR_CUDA;
  }
  *out = e;
  return LIO_OK;
}

extern "C" int lio_est_set_extrinsic(lio_est *e, const float tf7[7]) {
  if (!e || !tf7) return LIO_ERR_INVALID;
  for (int k = 0; k < 4; ++k) e->tlb_q[k] = tf7[k];
  for (int k = 0; k < 3; ++k) e->tlb_p[k] = tf7[4 + k];
  return LIO_OK;
}
extern "C" int lio_est_get_extrinsic(lio_est *e, float tf7[7]) {
  if (!e || !tf7) return LIO_ERR_INVALID;
  for (int k = 0; k < 4; ++k) tf7[k] = e->tlb_q[k];
  for (int k = 0; k < 3; ++k) tf7[4 + k] = e->tlb_p[k];
  return LIO_OK;
}

extern "C" int lio_est_init_frame(lio_est *e, int k, const double s[16], const float *surf_ds, int n, lio_pim *pim) {
  if (!e || !s || k < 0 || k >= e->W || n < 0 || (n > 0 && !surf_ds)) return LIO_ERR_INVALID;
  if (n > e->cfg.max_frame_points) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  e->Ps[k] = V3(s); e->Rs[k] = toR(normalized(Q(s[6], s[3], s[4], s[5]))); e->Vs[k] = V3(s + 7); e->Bas[k] = V3(s + 10); e->Bgs[k] = V3(s + 13);
  const int slot = e->slot_of[k + 1];  // one slot to the right: the first process_scan pushes (see oracle InitFrame)
  if (n > 0) LIO_CUDA_OK(cudaMemcpyAsync(e->slot_ptr[slot], surf_ds, sizeof(float4) * n, cudaMemcpyHostToDevice, e->stream));
  LIO_CUDA_OK(cudaMemcpyAsync(e->d_slot_n + slot, &n, sizeof(int), cudaMemcpyHostToDevice, e->stream));
  LIO_CUDA_OK(cudaMemcpyAsync(e->d_own_n + slot, &n, sizeof(int), cudaMemcpyHostToDevice, e->stream));
  LIO_CUDA_OK(cudaStreamSynchronize(e->stream));
  e->size_surf_stack[k + 1] = n;
  e->pre[k + 1] = pim ? pim->p : nullptr;
  if (pim) delete pim;
  return LIO_OK;
}

extern "C" int lio_est_finish_init(lio_est *e, const double a[3], const double g[3]) {
  if (!e || !a || !g) return LIO_ERR_INVALID;
  const int W = e->W;
  e->Ps[W] = e->Ps[W - 1]; e->Rs[W] = e->Rs[W - 1]; e->Vs[W] = e->Vs[W - 1]; e->Bas[W] = e->Bas[W - 1]; e->Bgs[W] = e->Bgs[W - 1];
  e->acc_last = V3(a); e->gyr_last = V3(g);
  e->first_imu = true;
  e->tmp_pre = std::make_shared<Preintegration>(e->acc_last, e->gyr_last, e->Bas[W], e->Bgs[W], e->noise);
  e->imu_stamped.clear();
  return LIO_OK;
}

extern "C" int lio_est_process_imu(lio_est *e, double dt, const double a[3], const double g[3], double stamp) {
  if (!e || !a || !g) return LIO_ERR_INVALID;
  const V3 acc(a), gyr(g);
  if (!e->first_imu) { e->first_imu = true; e->acc_last = acc; e->gyr_last = gyr; }
  if (!e->tmp_pre) return LIO_ERR_INVALID;
  const int j = e->W;
  e->tmp_pre->push_back(dt, acc, gyr);
  const V3 un_acc_0 = e->Rs[j] * (e->acc_last - e->Bas[j]) + e->g_vec;
  const V3 un_gyr = 0.5 * (e->gyr_last + gyr) - e->Bgs[j];
  e->Rs[j] = e->Rs[j] * toR(deltaQ(un_gyr * dt));
  const V3 un_acc_1 = e->Rs[j] * (acc - e->Bas[j]) + e->g_vec;
  const V3 un_acc = 0.5 * (un_acc_0 + un_acc_1);
  e->Ps[j] = e->Ps[j] + dt * e->Vs[j] + 0.5 * dt * dt * un_acc;
  e->Vs[j] = e->Vs[j] + dt * un_acc;
  ImuStampedF tt;
  tt.time = stamp;
  tt.p[0] = (float)e->Ps[j].x; tt.p[1] = (float)e->Ps[j].y; tt.p[2] = (float)e->Ps[j].z;
  {  // Quaternionf(Rs.cast<float>())
    M3 Rf;
    for (int a2 = 0; a2 < 3; ++a2) for (int b = 0; b < 3; ++b) Rf(a2, b) = (double)(float)e->Rs[j](a2, b);
    Q q = fromR(Rf);
    tt.q[0] = (float)q.x; tt.q[1] = (float)q.y; tt.q[2] = (float)q.z; tt.q[3] = (float)q.w;
  }
  e->imu_stamped.push_back(tt);
  if (e->imu_stamped.size() > 100) e->imu_stamped.erase(e->imu_stamped.begin());
  e->acc_last = acc; e->gyr_last = gyr;
  return LIO_OK;
}

extern "C" int lio_est_process_imu_batch(lio_est *e, int n, const double *dt, const double *acc3, const double *gyr3, const double *stamp) {
  if (!e || n < 0 || (n > 0 && (!dt || !acc3 || !gyr3 || !stamp))) return LIO_ERR_INVALID;
  for (int k = 0; k < n; ++k) {
    const int rc = lio_est_process_imu(e, dt[k], acc3 + 3 * k, gyr3 + 3 * k, stamp[k]);
    if (rc != LIO_OK) return rc;
  }
  return LIO_OK;
}

// ---- parameter <-> state ---------------------------------------------------------------------------
static void vector_to_double(lio_est *e) {  // Estimator.cc:2440-2478
  const int pivot = e->W - e->O;
  for (int i = 0, oi = pivot; i <= e->O; ++i, ++oi) {
    double *pp = e->para_pose[i].data(), *sb = e->para_sb[i].data();
    pp[0] = e->Ps[oi].x; pp[1] = e->Ps[oi].y; pp[2] = e->Ps[oi].z;
    Q q = fromR(e->Rs[oi]);
    pp[3] = q.x; pp[4] = q.y; pp[5] = q.z; pp[6] = q.w;
    for (int k = 0; k < 3; ++k) { sb[k] = e->Vs[oi][k]; sb[3 + k] = e->Bas[oi][k]; sb[6 + k] = e->Bgs[oi][k]; }
  }
  e->para_ex[0] = e->tlb_p[0]; e->para_ex[1] = e->tlb_p[1]; e->para_ex[2] = e->tlb_p[2];
  e->para_ex[3] = e->tlb_q[0]; e->para_ex[4] = e->tlb_q[1]; e->para_ex[5] = e->tlb_q[2]; e->para_ex[6] = e->tlb_q[3];
  e->S_valid = false;
}

static void double_to_vector(lio_est *e) {  // Estimator.cc:2479-2568
  const int pivot = e->W - e->O, O = e->O;
  const V3 origin_P0 = e->Ps[pivot];
  const V3 origin_R0 = R2ypr(e->Rs[pivot]);
  auto qpose = [&](int i) { const double *p = e->para_pose[i].data(); return toR(normalized(Q(p[6], p[3], p[4], p[5]))); };
  const V3 origin_R00 = R2ypr(qpose(0));
  const double y_diff = origin_R0.x - origin_R00.x;
  M3 rot_diff = ypr2R(V3(y_diff, 0, 0));
  if (std::fabs(std::fabs(origin_R0.y) - 90) < 1.0 || std::fabs(std::fabs(origin_R00.y) - 90) < 1.0) rot_diff = e->Rs[pivot] * T(qpose(0));
  {
    Tw trans_pivot(fromR(e->Rs[pivot]), e->Ps[pivot]);
    Tw trans_opt_pivot(fromR(rot_diff * qpose(0)), origin_P0);
    for (int idx = 0; idx < pivot; ++idx) {
      Tw trans_idx(fromR(e->Rs[idx]), e->Ps[idx]);
      Tw o = tw_mul(tw_mul(trans_opt_pivot, tw_inverse(trans_pivot)), trans_idx);
      e->Ps[idx] = o.pos;
      e->Rs[idx] = toR(normalized(o.rot));
    }
  }
  for (int i = 0, oi = pivot; i <= O; ++i, ++oi) {
    const double *pp = e->para_pose[i].data(), *p0 = e->para_pose[0].data(), *sb = e->para_sb[i].data();
    e->Rs[oi] = rot_diff * qpose(i);
    e->Ps[oi] = rot_diff * V3(pp[0] - p0[0], pp[1] - p0[1], pp[2] - p0[2]) + origin_P0;
    e->Vs[oi] = rot_diff * V3(sb[0], sb[1], sb[2]);
    e->Bas[oi] = V3(sb[3], sb[4], sb[5]);
    e->Bgs[oi] = V3(sb[6], sb[7], sb[8]);
  }
  e->tlb_p[0] = (float)e->para_ex[0]; e->tlb_p[1] = (float)e->para_ex[1]; e->tlb_p[2] = (float)e->para_ex[2];
  e->tlb_q[0] = (float)e->para_ex[3]; e->tlb_q[1] = (float)e->para_ex[4]; e->tlb_q[2] = (float)e->para_ex[5]; e->tlb_q[3] = (float)e->para_ex[6];
}

// ---- stage B orchestration -----------------------------------------------------------------------
extern "C" int lio_est_frame_owner(int frame_rel, int world);
// ranks the lidar reduction of a solve is sharded over: 1 when the features themselves were exchanged (every rank holds all of them)
static int solve_world(const lio_est *e) { return e->fpeers ? 1 : e->world; }
static bool owns_frame(const lio_est *e, int idx) {  // idx: logical frame > pivot
  const int pivot = e->W - e->O;
  return lio_est_frame_owner(idx - pivot, e->world) == e->rank;
}

__global__ void k_xwait(const unsigned *__restrict__ flags, int npeers, unsigned epoch, int *__restrict__ err, const int *__restrict__ skip);

static int build_local_map(lio_est *e, const std::function<int()> &before_sync = nullptr) {
  const int W = e->W, O = e->O, pivot = W - O;
  cudaStream_t st = e->stream;
  const double t0 = now_s();
  const Tw tlb = tlb_double(e);
  const Tw transform_pivot = lidar_pose(e->Ps[pivot], e->Rs[pivot], tlb);
  const Tw pivot_inv = tw_inverse(transform_pivot);
  if (!e->init_local_map) {  // :1409-1441 merge frames 0..pivot into the pivot cloud
    if (pivot > 0) {
      ConcatParams cp;
      std::memset(&cp, 0, sizeof(cp));
      cp.nsrc = pivot + 1;
      for (int i = 0; i <= pivot; ++i) {
        AffineF a = to_affine_f(tw_mul(pivot_inv, lidar_pose(e->Ps[i], e->Rs[i], tlb)));
        cp.src[i] = e->slot_ptr[e->slot_of[i]];
        cp.n[i] = e->d_slot_n + e->slot_of[i];
        std::memcpy(cp.R[i], a.R, sizeof(a.R)); std::memcpy(cp.t[i], a.t, sizeof(a.t));
        cp.tag[i] = -1.f;  // keep intensity
      }
      k_concat<<<std::max(1, std::min(e->sm_count * 2, (e->slot_cap + 255) / 256)), 256, 0, st>>>(cp, e->d_tmp, e->d_counts + 3, e->slot_cap);
      ++e->launches;
      const int ps = e->slot_of[pivot];
      EST_CUDA(cudaMemcpyAsync(e->slot_ptr[ps], e->d_tmp, sizeof(float4) * e->slot_cap, cudaMemcpyDeviceToDevice, st));
      EST_CUDA(cudaMemcpyAsync(e->d_slot_n + ps, e->d_counts + 3, sizeof(int), cudaMemcpyDeviceToDevice, st));
    }
    e->init_local_map = true;
  }
  ConcatParams cp;
  std::memset(&cp, 0, sizeof(cp));
  int ns = 0;
  for (int i = 0; i <= W; ++i) {
    AffineF a = to_affine_f(tw_mul(pivot_inv, lidar_pose(e->Ps[i], e->Rs[i], tlb)));
    e->local_tf[i] = a.tf;
    e->h_tf[i] = a.tf;
    if (i < pivot || i == W) continue;
    cp.src[ns] = e->slot_ptr[e->slot_of[i]];
    cp.n[ns] = e->d_slot_n + e->slot_of[i];
    if (i == pivot) cp.identity[ns] = 1;
    else { std::memcpy(cp.R[ns], a.R, sizeof(a.R)); std::memcpy(cp.t[ns], a.t, sizeof(a.t)); cp.tag[ns] = (float)i; }
    ++ns;
  }
  cp.nsrc = ns;
  EST_CUDA(cudaMemcpyAsync(e->d_tf, e->h_tf, sizeof(TransformF) * (W + 1), cudaMemcpyHostToDevice, st));
  k_concat<<<std::max(1, std::min(e->sm_count * 4, (e->local_cap + 255) / 256)), 256, 0, st>>>(cp, e->d_local, e->d_counts + 1, e->local_cap);
  ++e->launches;
  // Host-side bound of the concatenated cloud: the frames' own sizes are mirrored on the host (the merged pivot cloud is
  // at most the sum of the frames merged into it), so the voxel grid, its sort and the hash build are sized for the data,
  // not for the worst-case capacity.
  long long bound = 64;
  for (int i = 0; i < W; ++i) bound += e->size_surf_stack[i] > 0 ? e->size_surf_stack[i] : e->cfg.max_frame_points;
  const int n_bound = (int)std::min<long long>(e->local_cap, bound);
  int rc = e->vg.run(e->d_local, e->d_counts + 1, n_bound, e->cfg.surf_filter_size, e->d_map, e->local_cap, e->d_counts + 2, nullptr, st, &e->launches);
  if (rc != LIO_OK) return rc;
  const float cell = std::sqrt(e->cfg.min_match_sq_dis) * (1.0f + 1.0f / 1024.0f);
  rc = e->hash.build(e->d_map, e->d_counts + 2, n_bound, cell, st, &e->launches);
  if (rc != LIO_OK) return rc;
  e->t_build = now_s() - t0;
  const double t1 = now_s();
  if (e->fpeers) {
    // feature exchange: this scan's features go to the other parity (a rank that is one scan ahead writes into the parity nobody
    // reads any more); only the counts of the frames this rank matches are reset - the others arrive from their owners
    set_feature_parity(e, e->fparity ^ 1);
    ++e->fepoch;
    for (int idx = pivot + 1; idx <= W; ++idx)
      if (owns_frame(e, idx)) EST_CUDA(cudaMemsetAsync(e->d_feat_counts + idx, 0, sizeof(int), st));
  } else {
    EST_CUDA(cudaMemsetAsync(e->d_feat_counts, 0, sizeof(int) * (W + 1), st));
  }
  // CalculateLaserOdom on the newest frame: rounds after convergence are no-ops on the device (done flag), but each still costs two
  // launches.  The chain is therefore enqueued in two batches: the first kOdomFirstBatch rounds ride with the scan's one
  // synchronisation (it converges in 2-3 rounds); only if the flag is still clear are the remaining rounds enqueued.
  constexpr int kOdomFirstBatch = 3;
  const bool odom = e->cfg.imu_factor && owns_frame(e, W);
  KnnBatch ob;
  auto odom_rounds = [&](int from, int to, cudaStream_t q) -> int {
    const int idx = W, slot = e->slot_of[W];
    if (!e->cfg.keep_features) {
      // two launches per round and no memset: the k-NN + plane fit of the newest frame, then ONE CTA that reduces the
      // round's features to A^T A / A^T b, takes the 6 x 6 Gauss-Newton step and re-arms the k-NN launch state
      ob.nframes = 1;
      KnnFrame &f = ob.f[0];
      f.surf = e->slot_ptr[slot]; f.n_dev = e->d_slot_n + slot; f.n_bound = e->cfg.max_frame_points; f.tf = e->d_tf + idx;
      f.out_p = e->feats[idx].pts; f.out_c = e->feats[idx].coef; f.out_src = e->feats[idx].src; f.out_count = e->feats[idx].count;
      f.append = 0; f.tile0 = 0;
      for (int it = from; it < to; ++it) {
        int r2 = calculate_features_batch(e->hash, ob, e->cfg.min_match_sq_dis, e->cfg.min_plane_dis, &e->d_odom->done, e->knn2, q, &e->launches,
                                          0, it > 0);
        if (r2 != LIO_OK) return r2;
        k_odom_round<<<1, kOdomRoundThreads, 0, q>>>(e->feats[idx].pts, e->feats[idx].coef, e->feats[idx].count, e->d_tf + idx, e->d_odom, 0.05, 0.05,
                                                      e->knn2.status, ob.ntiles, e->knn2.ticket);
        ++e->launches;
      }
    } else {
      // keep_features: every round re-evaluates ALL kept features at the current transform (Estimator.cc:978-980), so the
      // reduction is a pass of its own
      const int nb = std::max(1, std::min(e->sm_count, (e->feats[idx].cap + kOdomThreads - 1) / kOdomThreads));
      for (int it = from; it < to; ++it) {
        int r2 = calculate_features_dev(e->hash, e->d_map, e->slot_ptr[slot], e->d_slot_n + slot, e->cfg.max_frame_points, e->d_tf + idx,
                                        e->cfg.min_match_sq_dis, e->cfg.min_plane_dis, e->feats[idx], 1,
                                        &e->d_odom->done, e->knn2, q, &e->launches);
        if (r2 != LIO_OK) return r2;
        k_odom_reduce<<<nb, kOdomThreads, 0, q>>>(e->feats[idx].pts, e->feats[idx].coef, e->feats[idx].count, e->d_tf + idx, e->d_odom, e->d_odom_partial);
        k_odom_solve<<<1, 32, 0, q>>>(e->d_odom, e->d_tf + idx, 0.05, 0.05);
        e->launches += 2;
      }
    }
    return LIO_OK;
  };
  const int odom_total = odom ? e->cfg.odom_max_iterations : 0;
  const int odom_first = e->fpeers ? odom_total : std::min(odom_total, kOdomFirstBatch);   // exchanged features must be final
  if (odom) {
    // the chain is a string of small latency-bound launches: it runs on its own stream beside the frame-batched launch below
    // (both only read the map and its hash; the feature buffers are per frame) and joins before the read-back
    EST_CUDA(cudaEventRecord(e->ev_map, st));
    EST_CUDA(cudaStreamWaitEvent(e->ostream, e->ev_map, 0));
    EST_CUDA(cudaMemsetAsync(e->d_odom, 0, sizeof(OdomState), e->ostream));
    rc = odom_rounds(0, odom_first, e->ostream);
    if (rc != LIO_OK) return rc;
    EST_CUDA(cudaEventRecord(e->ev_odom, e->ostream));
  }
  {
    // every owned frame except a LaserOdom-driven newest frame: ONE batched kNN + plane-fit launch
    KnnBatch b;
    b.nframes = 0;
    for (int idx = pivot + 1; idx <= W; ++idx) {
      if (!owns_frame(e, idx)) continue;
      if (idx == W && e->cfg.imu_factor) continue;
      const int slot = e->slot_of[idx];
      KnnFrame &f = b.f[b.nframes++];
      f.surf = e->slot_ptr[slot]; f.n_dev = e->d_slot_n + slot; f.tf = e->d_tf + idx;
      const int known = e->size_surf_stack[idx];
      f.n_bound = (known > 0 && idx < W) ? known : e->cfg.max_frame_points;
      f.out_p = e->feats[idx].pts; f.out_c = e->feats[idx].coef; f.out_src = e->feats[idx].src; f.out_count = e->feats[idx].count;
      f.append = 0; f.tile0 = 0;
    }
    e->knn_timed = b.nframes > 0 && e->evk0 && e->evk1;
    if (e->knn_timed) cudaEventRecord(e->evk0, st);
    rc = calculate_features_batch(e->hash, b, e->cfg.min_match_sq_dis, e->cfg.min_plane_dis, nullptr, e->knn, st, &e->launches);
    if (rc != LIO_OK) return rc;
    if (e->knn_timed) cudaEventRecord(e->evk1, st);
  }
  // one synchronisation: feature counts, map size, odom iterations
  auto readback = [&]() -> int {
    EST_CUDA(cudaMemcpyAsync(e->h_counts, e->d_feat_counts, sizeof(int) * (W + 1), cudaMemcpyDeviceToHost, st));
    EST_CUDA(cudaMemcpyAsync(e->h_counts + W + 1, e->d_counts, sizeof(int) * 4, cudaMemcpyDeviceToHost, st));
    EST_CUDA(cudaMemcpyAsync(e->h_counts + W + 5, &e->d_odom->iter, sizeof(int), cudaMemcpyDeviceToHost, st));
    EST_CUDA(cudaMemcpyAsync(e->h_tf + W, e->d_tf + W, sizeof(TransformF), cudaMemcpyDeviceToHost, st));
    EST_CUDA(cudaMemcpyAsync(e->h_counts + W + 6, e->d_slot_n + e->slot_of[W], sizeof(int), cudaMemcpyDeviceToHost, st));
    EST_CUDA(cudaMemcpyAsync(e->h_counts + W + 7, e->vg.overflow_flag(), sizeof(int), cudaMemcpyDeviceToHost, st));
    EST_CUDA(cudaMemcpyAsync(e->h_counts + W + 8, &e->d_odom->done, sizeof(int), cudaMemcpyDeviceToHost, st));
    if (e->fpeers) EST_CUDA(cudaMemcpyAsync(e->h_counts + W + 9, e->fslab + e->foff_flags + 128, sizeof(int), cudaMemcpyDeviceToHost, st));
    EST_CUDA(cudaStreamSynchronize(st));
    return LIO_OK;
  };
  if (odom) EST_CUDA(cudaStreamWaitEvent(st, e->ev_odom, 0));
  if (e->fpeers) {
    // all-gather of the features: every owned frame is copied into the same place of every peer's slab, then the scan's epoch is
    // published in every rank's flag slot and this rank waits for the epochs of all ranks (bounded, like the S-row exchange)
    const size_t pbase = (size_t)e->fparity * e->fpar_stride;
    FeaturePeers fp;
    std::memset(&fp, 0, sizeof(fp));
    fp.npeers = e->world; fp.self = e->rank;
    FlagPeers fl;
    std::memset(&fl, 0, sizeof(fl));
    fl.npeers = e->world; fl.self = e->rank;
    for (int r = 0; r < e->world; ++r) fl.flag[r] = reinterpret_cast<unsigned *>(e->fpeer_base[r] + e->foff_flags);
    for (int idx = pivot + 1; idx <= W; ++idx) {
      if (!owns_frame(e, idx)) continue;
      for (int r = 0; r < e->world; ++r) {
        fp.pts[r] = reinterpret_cast<float4 *>(e->fpeer_base[r] + pbase + e->foff_pts[idx]);
        fp.coef[r] = reinterpret_cast<float4 *>(e->fpeer_base[r] + pbase + e->foff_coef[idx]);
        fp.count[r] = reinterpret_cast<int *>(e->fpeer_base[r] + pbase + e->foff_cnt) + idx;
      }
      const int known = e->size_surf_stack[idx];
      const int bound = (known > 0 && idx < W) ? known : e->feats[idx].cap;
      k_publish_features<<<std::max(1, std::min(e->sm_count * 2, (bound + 255) / 256)), 256, 0, st>>>(e->feats[idx].pts, e->feats[idx].coef, e->feats[idx].count,
                                                                                                   e->feats[idx].cap, fp);
      ++e->launches;
    }
    k_publish_flag<<<1, 32, 0, st>>>(fl, e->fepoch);
    k_xwait<<<1, 32, 0, st>>>(reinterpret_cast<const unsigned *>(e->fslab + e->foff_flags), e->world, e->fepoch,
                              reinterpret_cast<int *>(e->fslab + e->foff_flags + 128), nullptr);
    e->launches += 2;
  }
  if (before_sync) {   // host work that only needs the window state runs here, while the GPU is busy with the launches above
    rc = before_sync();
    if (rc != LIO_OK) return rc;
  }
  rc = readback();
  if (rc != LIO_OK) return rc;
  if (odom && odom_first < odom_total && !e->h_counts[W + 8]) {   // not converged yet (rare): the rest of the chain, one more synchronisation
    rc = odom_rounds(odom_first, odom_total, st);
    if (rc != LIO_OK) return rc;
    rc = readback();
    if (rc != LIO_OK) return rc;
  }
  if (e->fpeers && e->h_counts[W + 9]) {
    cudaMemsetAsync(e->fslab + e->foff_flags + 128, 0, sizeof(int), st);
    lio_set_last_error(__FILE__, __LINE__, "feature exchange timed out (a rank did not publish its frames)");
    return LIO_ERR_CUDA;
  }
  if (e->h_counts[W + 6] > e->cfg.max_frame_points) {   // vg_emit stopped storing at the capacity but kept counting
    lio_set_last_error(__FILE__, __LINE__, "down-sampled scan exceeds max_frame_points");
    return LIO_ERR_CAPACITY;
  }
  if (e->h_counts[W + 7]) {   // PCL: "Leaf size is too small for the input dataset. Integer indices would overflow."
    cudaMemsetAsync(e->vg.overflow_flag(), 0, sizeof(int), st);
    lio_set_last_error(__FILE__, __LINE__, "voxel grid index overflow (leaf size too small for the cloud extent)");
    return LIO_ERR_CAPACITY;
  }
  e->size_surf_stack[W] = e->h_counts[W + 6];
  if (e->knn_timed) {  // live duration of the frame-batched k-NN + plane-fit launch (its memsets included, ~2 us)
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->evk0, e->evk1) == cudaSuccess) {
      long long nq = 0;
      for (int idx = pivot + 1; idx <= W; ++idx)
        if (owns_frame(e, idx) && !(idx == W && e->cfg.imu_factor)) nq += e->size_surf_stack[idx];
      e->knn_ms_sum += ms; e->knn_launch_count += 1; e->knn_query_sum += nq;
    }
  }
  for (int k = 0; k <= W; ++k) e->h_feat_n[k] = e->h_counts[k];
  e->h_map_n = e->h_counts[W + 1 + 2];
  e->odom_iters = e->h_counts[W + 5];
  e->local_tf[W] = e->h_tf[W];
  for (int k = pivot + 1; k <= W; ++k)
    if (e->h_feat_n[k] > e->feats[k].cap) { lio_set_last_error(__FILE__, __LINE__, "feature buffer overflow"); return LIO_ERR_CAPACITY; }
  if (e->h_counts[W + 1 + 1] >= e->local_cap) { lio_set_last_error(__FILE__, __LINE__, "local map capacity exceeded"); return LIO_ERR_CAPACITY; }
  if (e->h_counts[W + 1 + 1] > n_bound) { lio_set_last_error(__FILE__, __LINE__, "internal: host bound of the local cloud below its device count"); return LIO_ERR_CAPACITY; }
  e->t_feat = now_s() - t1;
  return LIO_OK;
}

// ---- fused exchange over peer memory -----------------------------------------------------------------
// Waits until every rank has published `epoch` in this rank's flag array (the rows travel with the asm_ppp tails of the
// peers as P2P stores; system-scope release / acquire).  Bounded: a peer that never arrives sets *err instead of hanging.
__global__ void k_xwait(const unsigned *__restrict__ flags, int npeers, unsigned epoch, int *__restrict__ err,
                        const int *__restrict__ skip) {
  const int p = threadIdx.x;
  if (p >= npeers) return;
  if (skip && *skip) return;   // the device solver has terminated: its asm_ppp launches publish nothing any more
  const long long t0 = clock64();
  while (true) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + p) : "memory");
    if ((int)(v - epoch) >= 0) break;
    if (clock64() - t0 > 20000000000LL) { *err = 1; break; }   // ~10 s at 1.97 GHz
    __nanosleep(64);
  }
}

// ---- stage C: lidar reduction at the current parameter values ------------------------------------
struct FrameTerms { double R[9], t[3], M[6 * 18]; };

static int eval_lidar_wait(lio_est *e);
// Enqueues the fused lidar reduction at the current parameters (no host synchronisation); eval_lidar_wait() completes it.
static int eval_lidar_launch(lio_est *e, std::vector<FrameTerms> &ft) {
  const int O = e->O, pivot = e->W - O;
  ft.resize(O + 1);
  AsmParams ap;
  std::memset(&ap, 0, sizeof(ap));
  ap.nframes = O;
  for (int i = 1; i <= O; ++i) {
    ppp_frame_terms(e->para_pose[0].data(), e->para_pose[i].data(), e->para_ex, ft[i].R, ft[i].t, ft[i].M);
    AsmFrame &f = ap.f[i - 1];
    const FeatureOut &fo = e->feats[pivot + i];
    f.pts = fo.pts; f.coef = fo.coef;
    f.n = (e->cfg.point_distance_factor && (e->fpeers || owns_frame(e, pivot + i))) ? e->h_feat_n[pivot + i] : 0;
    std::memcpy(e->h_Rt + (i - 1) * kAsmRtStride, ft[i].R, sizeof(double) * 9);
    std::memcpy(e->h_Rt + (i - 1) * kAsmRtStride + 9, ft[i].t, sizeof(double) * 3);
  }
  if (e->S_valid) return LIO_OK;
  EST_CUDA(cudaMemcpyAsync(e->d_Rt, e->h_Rt, sizeof(double) * O * kAsmRtStride, cudaMemcpyHostToDevice, e->stream));
  asm_plan(ap, e->sm_count);
  long long nfeat = 0;
  for (int k = 0; k < ap.nframes; ++k) nfeat += ap.f[k].n;
  const bool peers = solve_world(e) > 1 && e->npeers == e->world;
  if (solve_world(e) > 1 && !peers && !e->allreduce) {
    lio_set_last_error(__FILE__, __LINE__, "sharded context without an exchange: call lio_est_set_peers or pass an allreduce callback");
    return LIO_ERR_INVALID;
  }
  const double *result = e->asmw.out;
  if (peers) {  // the kernel's tail scatters the owned rows to every rank and publishes the epoch
    ap.npeers = e->npeers; ap.self = e->rank; ap.epoch = ++e->xepoch;
    const size_t par = (size_t)(ap.epoch & 1u) * kXRowBytes;
    for (int i = 1; i <= O; ++i) if (owns_frame(e, pivot + i)) ap.owned_mask |= 1u << (i - 1);
    for (int r = 0; r < e->npeers; ++r) {
      ap.peer_out[r] = reinterpret_cast<double *>(e->peer_base[r] + par);
      ap.peer_flag[r] = reinterpret_cast<unsigned *>(e->peer_base[r] + kXFlagOff);
    }
    result = reinterpret_cast<const double *>(e->xbuf + par);
  }
  if (e->ev0) cudaEventRecord(e->ev0, e->stream);
  int rc = asm_launch(ap, e->d_Rt, e->asmw, e->stream, &e->launches);
  if (rc != LIO_OK) return rc;
  if (e->ev1) cudaEventRecord(e->ev1, e->stream);
  if (peers) {
    k_xwait<<<1, 32, 0, e->stream>>>(reinterpret_cast<const unsigned *>(e->xbuf + kXFlagOff), e->npeers, ap.epoch,
                                     reinterpret_cast<int *>(e->xbuf + kXErrOff), nullptr);
    ++e->launches;
    EST_CUDA(cudaMemcpyAsync(e->h_S + kMaxOpt * kAsmStride, e->xbuf + kXErrOff, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  } else if (solve_world(e) > 1 && e->allreduce) {
    rc = e->allreduce(e->allreduce_user, e->asmw.out, O * kAsmStride);
    if (rc != 0) { lio_set_last_error(__FILE__, __LINE__, "allreduce callback failed"); return LIO_ERR_CUDA; }
  }
  EST_CUDA(cudaMemcpyAsync(e->h_S, result, sizeof(double) * O * kAsmStride, cudaMemcpyDeviceToHost, e->stream));
  e->S_pending = true;
  e->S_pending_feats = nfeat;
  return LIO_OK;
}

static int eval_lidar_wait(lio_est *e) {
  if (!e->S_pending) return LIO_OK;
  const double t0 = now_s();
  EST_CUDA(cudaStreamSynchronize(e->stream));
  e->t_lin_wait += now_s() - t0;
  e->S_pending = false;
  if (*reinterpret_cast<const int *>(e->h_S + kMaxOpt * kAsmStride)) {
    cudaMemsetAsync(e->xbuf + kXErrOff, 0, sizeof(int), e->stream);   // the flag is one-shot: clear it with the report
    *reinterpret_cast<int *>(e->h_S + kMaxOpt * kAsmStride) = 0;
    lio_set_last_error(__FILE__, __LINE__, "peer exchange timed out (a rank did not publish its rows)");
    return LIO_ERR_CUDA;
  }
  if (e->ev0 && e->ev1) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) == cudaSuccess) { e->asm_ms_sum += ms; e->asm_launch_count += 1; e->asm_feat_sum += e->S_pending_feats; }
  }
  e->S_valid = true;
  return LIO_OK;
}

static int eval_lidar(lio_est *e, std::vector<FrameTerms> &ft) {
  int rc = eval_lidar_launch(e, ft);
  return rc != LIO_OK ? rc : eval_lidar_wait(e);
}

// tangent layout: [pose_k(6) sb_k(9)] k=0..O, then ex(6)
static inline int off_pose(int k) { return 15 * k; }
static inline int off_sb(int k) { return 15 * k + 6; }

// adds M^T S M into H/g over (pose_0, pose_i, ex) column offsets o0, oi, oe (oe < 0: extrinsic not a variable)
static void add_lidar_block(const double *S /*kAsmStride*/, const double *M /*6x18*/, Mat *H, Vec *g, int o0, int oi, int oe) {
  double Sg[6][6], Sr[6];
  {
    int k = 0;
    for (int a = 0; a < 7; ++a) for (int b = a; b < 7; ++b) { double v = S[k++]; if (b < 6) { Sg[a][b] = v; Sg[b][a] = v; } else if (a < 6) Sr[a] = v; }
  }
  double SM[6][18];
  for (int a = 0; a < 6; ++a) for (int c = 0; c < 18; ++c) { double s = 0; for (int b = 0; b < 6; ++b) s += Sg[a][b] * M[b * 18 + c]; SM[a][c] = s; }
  const int offs[3] = {o0, oi, oe};
  for (int bi = 0; bi < 3; ++bi) {
    if (offs[bi] < 0) continue;
    for (int a = 0; a < 6; ++a) {
      const int ca = bi * 6 + a;
      double gs = 0;
      for (int k = 0; k < 6; ++k) gs += M[k * 18 + ca] * Sr[k];
      (*g)[offs[bi] + a] += gs;
      if (!H) continue;
      for (int bj = 0; bj < 3; ++bj) {
        if (offs[bj] < 0) continue;
        for (int b = 0; b < 6; ++b) {
          const int cb = bj * 6 + b;
          double s = 0;
          for (int k = 0; k < 6; ++k) s += M[k * 18 + ca] * SM[k][cb];
          (*H)(offs[bi] + a, offs[bj] + b) += s;
        }
      }
    }
  }
}

static void prior_dx(const lio_est *e, const MargPrior &pr, Vec &dx) {  // MarginalizationFactor::Evaluate :347-372
  const int O = e->O;
  dx.assign(pr.n, 0.0);
  auto pose_dx = [&](const double *x, const double *x0, double *out) {
    for (int k = 0; k < 3; ++k) out[k] = x[k] - x0[k];
    Q q0(x0[6], x0[3], x0[4], x0[5]), q(x[6], x[3], x[4], x[5]);
    Q dq = inverse(q0) * q;
    Q dn = normalized(dq);
    double s = dq.w < 0 ? -2.0 : 2.0;
    out[3] = s * dn.x; out[4] = s * dn.y; out[5] = s * dn.z;
  };
  for (int k = 0; k < O; ++k) {
    pose_dx(e->para_pose[k].data(), &pr.x0_pose[7 * k], &dx[15 * k]);
    for (int a = 0; a < 9; ++a) dx[15 * k + 6 + a] = e->para_sb[k][a] - pr.x0_sb[9 * k + a];
  }
  pose_dx(e->para_ex, pr.x0_ex, &dx[15 * O]);
}

// Drains the ImuFactor pool of the current linearisation (called concurrently by the caller thread and the helper).
static void imu_pool_run(lio_est *e, int O, int pivot) {
  int i;
  while ((i = e->imu_next.fetch_add(1)) < O) {
    lio_est::ImuBlockStore &b = e->imu_blocks_store[i];
    Preintegration &pim = *e->pre[pivot + i + 1];
    b.used = !(pim.sum_dt > 10.0);
    if (b.used) {
      double r[15], J[15][30];
      imu_factor_evaluate30(pim, e->para_pose[i].data(), e->para_sb[i].data(), e->para_pose[i + 1].data(), e->para_sb[i + 1].data(), r, J);
      JtJ_dense(&J[0][0], r, 15, 30, b.JtJ, b.Jtr);
      double sq = 0;
      for (int k = 0; k < 15; ++k) sq += r[k] * r[k];
      b.cost = 0.5 * sq;
    }
    e->imu_done.fetch_add(1);
  }
}

// Full linearisation at the current parameter values.  n_t = tangent dim (ex block present iff !ex_constant).
static bool linearize(lio_est *e, Mat &H, Vec &g, double &cost, double *c_pim, double *c_ppp, double *c_marg) {
  const int O = e->O, pivot = e->W - O;
  const bool ex_free = !e->ex_constant;
  const int n = 15 * (O + 1) + (ex_free ? 6 : 0);
  const int oe = ex_free ? 15 * (O + 1) : -1;
  std::vector<FrameTerms> ft;
  if (eval_lidar_launch(e, ft) != LIO_OK) return false;  // the device reduces the lidar factors while the host does the rest
  // H starts as the prior's information matrix scattered into the tangent layout (constant over a solve: cached), or zero
  const bool use_prior = e->cfg.marginalization_factor && e->prior.valid;
  if (use_prior) {
    if (!e->hp_exp_valid || e->hp_exp.r != n) {
      const MargPrior &pr = e->prior;
      e->hp_exp = Mat(n, n);
      const int nw = 15 * O;  // window part maps one to one, the extrinsic block moves behind pose_O / sb_O
      for (int a = 0; a < pr.n; ++a) {
        const int ta = a < nw ? a : (ex_free ? 15 * (O + 1) + (a - nw) : -1);
        if (ta < 0) continue;
        const double *row = &pr.Hp.d[(size_t)a * pr.n];
        double *hrow = &e->hp_exp.d[(size_t)ta * n];
        for (int b = 0; b < nw; ++b) hrow[b] = row[b];
        if (ex_free) for (int b = nw; b < pr.n; ++b) hrow[15 * (O + 1) + (b - nw)] = row[b];
      }
      e->hp_exp_valid = true;
    }
    if (H.r != n) H = Mat(n, n);
    std::memcpy(H.d.data(), e->hp_exp.d.data(), sizeof(double) * (size_t)n * n);
  } else {
    if (H.r != n) H = Mat(n, n); else H.zero();
  }
  g.assign(n, 0.0);
  const double th0 = now_s();
  double cp = 0, ci = 0, cm = 0;
  // ImuFactors: factors [0, i_split) go directly into H on this thread; factors [i_split, O) form a pool that the context's
  // helper thread and (after its own share and the prior) this thread drain together into private 30x30 blocks, which
  // are added in index order afterwards - the result does not depend on who evaluated which block, and a helper that
  // is late or descheduled costs nothing but its share.
  const int i_split = (e->cfg.imu_factor && O >= 4) ? O / 2 : O;
  auto imu_eval = [&](int i, double *r, double (*J)[30]) {
    Preintegration &pim = *e->pre[pivot + i + 1];
    if (pim.sum_dt > 10.0) return false;
    imu_factor_evaluate30(pim, e->para_pose[i].data(), e->para_sb[i].data(), e->para_pose[i + 1].data(), e->para_sb[i + 1].data(), r, J);
    return true;
  };
  if (e->cfg.imu_factor && i_split < O) {
    e->worker.wait();  // the previous pool job has retired before the counters are reset
    e->imu_next.store(i_split);
    e->imu_done.store(0);
    e->worker.submit([e, O, pivot]() { imu_pool_run(e, O, pivot); });
  }
  if (e->cfg.imu_factor) {
    for (int i = 0; i < i_split; ++i) {
      double r[15], J[15][30];
      if (!imu_eval(i, r, J)) continue;
      int cmap[30];
      for (int a = 0; a < 30; ++a) cmap[a] = 15 * i + a;  // pose_i, sb_i, pose_j, sb_j are contiguous in the tangent layout
      add_JtJ_mapped(&J[0][0], r, 15, 30, cmap, H, g);
      double sq = 0;
      for (int k = 0; k < 15; ++k) sq += r[k] * r[k];
      ci += 0.5 * sq;
    }
  }
  if (e->cfg.marginalization_factor && e->prior.valid) {
    const MargPrior &pr = e->prior;
    Vec dx;
    prior_dx(e, pr, dx);
    Vec Hdx;
    matvec(pr.Hp, dx, Hdx);
    cm = 0.5 * (pr.c0 + 2.0 * vdot(pr.bp, dx) + vdot(dx, Hdx));
    auto tmap = [&](int pi) { return pi < 15 * O ? pi : (ex_free ? 15 * (O + 1) + (pi - 15 * O) : -1); };
    for (int a = 0; a < pr.n; ++a) {
      const int ta = tmap(a);
      if (ta >= 0) g[ta] += Hdx[a] + pr.bp[a];
    }
  }
  if (e->cfg.imu_factor && i_split < O) {
    imu_pool_run(e, O, pivot);
    while (e->imu_done.load() < O - i_split) Worker::relax();  // at most one block still in flight on the helper
    const lio_est::ImuBlockStore *blk = e->imu_blocks_store;
    for (int i = i_split; i < O; ++i) {
      const lio_est::ImuBlockStore &b = blk[i];
      if (!b.used) continue;
      for (int a = 0; a < 30; ++a) {
        double *hrow = &H.d[(size_t)(15 * i + a) * n + 15 * i];
        const double *src = b.JtJ + 30 * a;
        for (int c = 0; c < 30; ++c) hrow[c] += src[c];
        g[15 * i + a] += b.Jtr[a];
      }
      ci += b.cost;
    }
  }
  double cprior = 0;
  if (e->cfg.prior_factor && ex_free) {  // constant extrinsic: the block is dropped from the reduced program
    const Tw tt = tlb_double(e);
    double r[6], J[6][6];
    prior_factor_evaluate(tt.pos, tt.rot, e->para_ex, r, J);
    for (int a = 0; a < 6; ++a) {
      double gs = 0;
      for (int k = 0; k < 6; ++k) gs += J[k][a] * r[k];
      g[oe + a] += gs;
      for (int b = 0; b < 6; ++b) { double s = 0; for (int k = 0; k < 6; ++k) s += J[k][a] * J[k][b]; H(oe + a, oe + b) += s; }
    }
    for (int k = 0; k < 6; ++k) cprior += 0.5 * r[k] * r[k];
  }
  e->t_lin_host += now_s() - th0;
  if (eval_lidar_wait(e) != LIO_OK) return false;
  if (e->cfg.point_distance_factor) {
    const double tl0 = now_s();
    for (int i = 1; i <= O; ++i) {
      const double *S = e->h_S + (i - 1) * kAsmStride;
      cp += 0.5 * S[28];
      add_lidar_block(S, ft[i].M, &H, &g, off_pose(0), off_pose(i), oe);
    }
    e->t_lin_lidar += now_s() - tl0;
  }
  cost = cp + ci + cm + cprior;
  if (c_pim) *c_pim = ci;
  if (c_ppp) *c_ppp = cp;
  if (c_marg) *c_marg = cm;
  return std::isfinite(cost);
}

static void prior_join(lio_est *e);
static int solve_dev_prepare(lio_est *e, int max_it, bool assemble_only);
static int slide_window(lio_est *e);
static MargPrior marg_algebra(Mat A, Vec b, int O, std::vector<double> x0_pose, std::vector<double> x0_sb, const double *x0_ex);
// ---- marginalisation (MarginalizationInfo::PreMarginalize / Marginalize, MarginalizationFactor.cc:132-311)
static int marginalize(lio_est *e) {
  const int O = e->O, pivot = e->W - O;
  const int m = 15, nr = 15 * O + 6, pos = m + nr;
  // layout: [pose_0 (6), sb_0 (9) | pose_1, sb_1, ..., pose_O, sb_O, ex]
  Mat A(pos, pos);
  Vec b(pos, 0.0);
  auto idx_pose = [&](int k) { return k == 0 ? 0 : m + 15 * (k - 1); };
  auto idx_sb = [&](int k) { return k == 0 ? 6 : m + 15 * (k - 1) + 6; };
  const int idx_ex = m + 15 * O;
  if (e->prior.valid) {  // previous prior re-wrapped with drop_set {pose_0, sb_0}
    const MargPrior &pr = e->prior;
    Vec dx;
    prior_dx(e, pr, dx);
    Vec Hdx;
    matvec(pr.Hp, dx, Hdx);
    auto map = [&](int pi) {  // prior canonical index -> A index
      if (pi >= 15 * O) return idx_ex + (pi - 15 * O);
      int k = pi / 15, a = pi % 15;
      return (a < 6 ? idx_pose(k) + a : idx_sb(k) + (a - 6));
    };
    for (int a = 0; a < pr.n; ++a) {
      const int ia = map(a);
      b[ia] += Hdx[a] + pr.bp[a];
      for (int c = 0; c < pr.n; ++c) A(ia, map(c)) += pr.Hp(a, c);
    }
  }
  if (e->cfg.imu_factor && e->pre[pivot + 1]->sum_dt < 10.0) {
    double r[15], J[15][30];
    imu_factor_evaluate30(*e->pre[pivot + 1], e->para_pose[0].data(), e->para_sb[0].data(), e->para_pose[1].data(), e->para_sb[1].data(), r, J);
    int col[30];
    for (int c = 0; c < 6; ++c) { col[c] = idx_pose(0) + c; col[15 + c] = idx_pose(1) + c; }
    for (int c = 0; c < 9; ++c) { col[6 + c] = idx_sb(0) + c; col[21 + c] = idx_sb(1) + c; }
    add_JtJ_mapped(&J[0][0], r, 15, 30, col, A, b);
  }
  if (e->cfg.point_distance_factor) {
    std::vector<FrameTerms> ft;
    int rc = eval_lidar(e, ft);
    if (rc != LIO_OK) return rc;
    for (int i = 1; i <= O; ++i) add_lidar_block(e->h_S + (i - 1) * kAsmStride, ft[i].M, &A, &b, idx_pose(0), idx_pose(i), idx_ex);
  }
  MargJob &job = e->mjob;
  job.O = O;
  job.A.r = A.r; job.A.c = A.c; job.A.d.swap(A.d);
  job.b.swap(b);
  job.x0_pose.resize(7 * O); job.x0_sb.resize(9 * O);
  for (int k = 1; k <= O; ++k) {  // addr_shift: block i -> i-1 in the next window
    std::memcpy(&job.x0_pose[7 * (k - 1)], e->para_pose[k].data(), 7 * sizeof(double));
    std::memcpy(&job.x0_sb[9 * (k - 1)], e->para_sb[k].data(), 9 * sizeof(double));
  }
  std::memcpy(job.x0_ex, e->para_ex, sizeof(job.x0_ex));
  job.stashed = true;
  if (!e->cfg.overlap_marginalization) {  // the reference's order: finish the algebra before returning from this scan
    job.stashed = false;
    e->prior = marg_algebra(std::move(job.A), std::move(job.b), job.O, std::move(job.x0_pose), std::move(job.x0_sb), job.x0_ex);
    e->hp_exp_valid = false;
  }
  return LIO_OK;
}

// Schur complement + eigen square-root form (MarginalizationInfo::Marginalize, MarginalizationFactor.cc:206-311) of a
// stashed system; layout [pose_0 (6), sb_0 (9) | pose_1, sb_1, ..., pose_O, sb_O, ex].  Pure function: worker-thread safe.
static MargPrior marg_algebra(Mat A, Vec b, int O, std::vector<double> x0_pose, std::vector<double> x0_sb, const double *x0_ex) {
  const int m = 15, nr = 15 * O + 6;
  // Schur complement with the eigen pseudo-inverse (eps = 1e-8)
  const double eps = 1e-8;
  Mat Amm(m, m);
  for (int r = 0; r < m; ++r) for (int c = 0; c < m; ++c) Amm(r, c) = 0.5 * (A(r, c) + A(c, r));
  Vec ev;
  Mat evec;
  sym_eigen(Amm, ev, evec);
  Mat Amm_inv(m, m);
  for (int r = 0; r < m; ++r)
    for (int c = 0; c < m; ++c) { double s = 0; for (int k = 0; k < m; ++k) s += evec(r, k) * (ev[k] > eps ? 1.0 / ev[k] : 0.0) * evec(c, k); Amm_inv(r, c) = s; }
  Mat Tm(nr, m);  // Arm * Amm_inv
  for (int r = 0; r < nr; ++r) for (int c = 0; c < m; ++c) { double s = 0; for (int k = 0; k < m; ++k) s += A(m + r, k) * Amm_inv(k, c); Tm(r, c) = s; }
  Mat A2(nr, nr);
  Vec b2(nr);
  for (int r = 0; r < nr; ++r) {
    for (int c = 0; c < nr; ++c) { double s = 0; for (int k = 0; k < m; ++k) s += Tm(r, k) * A(k, m + c); A2(r, c) = A(m + r, m + c) - s; }
    double s = 0;
    for (int k = 0; k < m; ++k) s += Tm(r, k) * b[k];
    b2[r] = b[m + r] - s;
  }
  // Eigen square root of the Schur complement (MarginalizationFactor.cc:276-311).  Only the factors that touch the dropped
  // blocks enter A, so the speed-bias blocks sb_2 .. sb_O (and pose_O's sb) have exactly-zero rows and columns in A2: its
  // spectrum is that of the non-zero principal sub-matrix plus zeros, which the eps test drops.  The decomposition is
  // therefore taken on the compressed matrix (75 of 156 rows for O = 10: ~9x fewer flops) and scattered back; the
  // reference decomposes the padded matrix and arrives at the same kept eigenpairs.
  std::vector<int> nz;
  for (int r = 0; r < nr; ++r) {
    bool any = b2[r] != 0.0;
    const double *row = &A2.d[(size_t)r * nr];
    for (int c = 0; c < nr && !any; ++c) any = row[c] != 0.0 || A2.d[(size_t)c * nr + r] != 0.0;
    if (any) nz.push_back(r);
  }
  const int nc = (int)nz.size();
  Mat Ac(nc, nc);
  Vec bc(nc);
  for (int r = 0; r < nc; ++r) {
    bc[r] = b2[nz[r]];
    for (int c = 0; c < nc; ++c) Ac(r, c) = A2(nz[r], nz[c]);
  }
  Vec ev2;
  Mat V2;
  if (nc > 0) sym_eigen(Ac, ev2, V2, 1);
  MargPrior np;
  np.valid = true;
  np.n = nr;
  np.Hp = Mat(nr, nr);
  np.bp.assign(nr, 0.0);
  np.c0 = 0;
  // Hp = V S V^T, bp = V_kept V_kept^T b, c0 = sum (v^T b)^2 / lambda over kept eigenpairs
  std::vector<int> kept;
  for (int k = 0; k < nc; ++k) if (ev2[k] > eps) kept.push_back(k);
  Vec vb(nc, 0.0);
  for (int k : kept) { double s = 0; for (int r = 0; r < nc; ++r) s += V2(r, k) * bc[r]; vb[k] = s; np.c0 += s * s / ev2[k]; }
  Mat Hc(nc, nc);
  if (nc > 0) weighted_gram(V2, ev2, kept, Hc);
  for (int r = 0; r < nc; ++r) {
    double sb = 0;
    for (int k : kept) sb += V2(r, k) * vb[k];
    np.bp[nz[r]] = sb;
    for (int c = 0; c < nc; ++c) np.Hp(nz[r], nz[c]) = Hc(r, c);
  }
  np.x0_pose = std::move(x0_pose);
  np.x0_sb = std::move(x0_sb);
  std::memcpy(np.x0_ex, x0_ex, sizeof(np.x0_ex));
  return np;
}

static void marg_start(lio_est *e) {
  MargJob &job = e->mjob;
  if (!job.stashed || job.running) return;
  job.stashed = false;
  job.running = true;
  e->worker.submit([&job]() {
    job.result = marg_algebra(std::move(job.A), std::move(job.b), job.O, std::move(job.x0_pose), std::move(job.x0_sb), job.x0_ex);
  });
}

// Makes e->prior current: runs a stashed job (inline start) and waits for a running one.
static void prior_join(lio_est *e) {
  MargJob &job = e->mjob;
  if (job.stashed) marg_start(e);
  if (!job.running) return;
  const double t0 = now_s();
  e->worker.wait();
  e->prior = std::move(job.result);
  e->hp_exp_valid = false;
  job.running = false;
  e->t_marg_wait += now_s() - t0;
}

// SolveOptimization (Estimator.cc:1648-2438) in three phases, also exported one by one (lio_est_open_scan_* / lio_est_solve /
// lio_est_close_scan) for callers that keep the reference's control flow:
//   scan_open   BuildLocalMap, join the previous marginalisation, VectorToDouble                       (:1361-1646, :2440-2478)
//   scan_solve  problem build + gates + ceres::Solve from the para_* blocks                            (:1747-1990)
//   scan_close  DoubleToVector, marginalisation of the oldest frame, SlideWindow                        (:2479-2568, :2040-2275, :2570-2666)
static int scan_open_window(lio_est *e) {
  e->turn_off = true;
  e->ds_prepared = false;
  int rc = build_local_map(e, [e]() -> int {
    prior_join(e);  // the previous scan's marginalisation algebra ran beside the front end enqueued above
    e->ex_constant = (e->extrinsic_stage == 0 || e->cfg.opt_extrinsic == 0);
    vector_to_double(e);
    // the device solver's state does not depend on the features: prepare and upload it before waiting for them
    if (e->use_dev_solver) return solve_dev_prepare(e, e->cfg.max_num_iterations, false);
    return LIO_OK;
  });
  if (rc != LIO_OK) return rc;
  e->window_open = true;
  return LIO_OK;
}

static int solve_host(lio_est *e, int max_it) {
  const int O = e->O;
  const double t0 = now_s();
  // residuals before optimisation + gates (:1924-1985)
  Mat H;
  Vec g;
  double cost;
  if (!linearize(e, H, g, cost, &e->cost_pim, &e->cost_ppp, &e->cost_marg)) { lio_set_last_error(__FILE__, __LINE__, "non-finite cost at the initial point"); return LIO_ERR_NUMERIC; }
  if (e->cfg.imu_factor) e->turn_off = e->cost_pim > 1e3;
  const bool ex_constant_before = e->ex_constant, prior_before = e->prior.valid;
  {
    const double ratio = e->cost_marg / (e->cost_ppp + e->cost_pim);
    if (!e->convergence_flag && !e->turn_off && ratio <= 2 && ratio != 0) e->convergence_flag = true;
    if (!e->convergence_flag) {
      e->ex_constant = true;
      e->prior.valid = false;
    }
  }
  DoglegProblem P;
  const bool ex_free = !e->ex_constant;
  P.n = 15 * (O + 1) + (ex_free ? 6 : 0);
  bool first = true;
  // the gate evaluation above is the solver's first linearisation when the gates left the problem structure unchanged
  bool reuse_gate = (ex_constant_before == e->ex_constant && prior_before == e->prior.valid);
  P.linearize = [&](Mat &Hh, Vec &gg, double &c) {
    bool ok = true;
    if (reuse_gate && first) { Hh.d.swap(H.d); Hh.r = H.r; Hh.c = H.c; gg.swap(g); c = cost; }
    else ok = linearize(e, Hh, gg, c, nullptr, nullptr, nullptr);
    if (ok && first) { e->H0 = Hh; e->g0 = gg; e->cost0 = c; e->have_H0 = true; first = false; }
    return ok;
  };
  P.get_state = [&](Vec &x) {
    x.clear();
    for (int k = 0; k <= O; ++k) { x.insert(x.end(), e->para_pose[k].begin(), e->para_pose[k].end()); x.insert(x.end(), e->para_sb[k].begin(), e->para_sb[k].end()); }
    if (ex_free) x.insert(x.end(), e->para_ex, e->para_ex + 7);
  };
  P.set_state = [&](const Vec &x) {
    for (int k = 0; k <= O; ++k) { std::memcpy(e->para_pose[k].data(), &x[16 * k], 7 * sizeof(double)); std::memcpy(e->para_sb[k].data(), &x[16 * k + 7], 9 * sizeof(double)); }
    if (ex_free) std::memcpy(e->para_ex, &x[16 * (O + 1)], 7 * sizeof(double));
    e->S_valid = false;
  };
  P.plus = [&](const Vec &x, const Vec &d, Vec &out) {
    out = x;
    for (int k = 0; k <= O; ++k) {
      pose_plus(&x[16 * k], &d[15 * k], &out[16 * k]);
      for (int a = 0; a < 9; ++a) out[16 * k + 7 + a] = x[16 * k + 7 + a] + d[15 * k + 6 + a];
    }
    if (ex_free) pose_plus(&x[16 * (O + 1)], &d[15 * (O + 1)], &out[16 * (O + 1)]);
  };
  DoglegOptions opt;
  opt.max_num_iterations = max_it;
  dogleg_solve(opt, P, &e->summary);
  if (e->summary.termination == 2 && !std::isfinite(e->summary.final_cost)) { lio_set_last_error(__FILE__, __LINE__, "solver breakdown"); return LIO_ERR_NUMERIC; }
  e->t_solve = now_s() - t0;
  return LIO_OK;
}

static int scan_close_window(lio_est *e) {
  double_to_vector(e);
  const double t1 = now_s();
  if (e->cfg.marginalization_factor && !e->turn_off) {
    vector_to_double(e);
    const int rc = marginalize(e);
    if (rc != LIO_OK) return rc;
    e->prior_uploaded = false;
  }
  e->t_marg = now_s() - t1;
  e->window_open = false;
  return slide_window(e);
}

// ---- SolveOptimization with the device-resident dogleg loop --------------------------------------
// The solve from the current para_* blocks on the device.  assemble_only: one evaluation without gates or steps, nothing of
// the estimator's own state is touched (lio_est_assemble); the first linearisation stays readable in ds.H0 / ds.g0.
// Everything of a device solve that does not depend on this scan's features: the solver state (parameters, prior, pre-integrations)
// and the frame terms of the initial point, uploaded asynchronously.  process_scan calls it while the GPU is still busy with the front
// end (before the scan's one synchronisation); solve_dev repeats it only when the parameters were replaced since.
static int solve_dev_prepare(lio_est *e, int max_it, bool assemble_only) {
  const int O = e->O, pivot = e->W - O;
  cudaStream_t st = e->stream;
  DevSolveState &S = *e->ds.h_st;
  S.sc.O = O; S.sc.n = 15 * (O + 1) + 6; S.sc.max_it = assemble_only ? 0 : max_it;
  S.sc.skip_gates = assemble_only ? 1 : 0; S.sc.pad_ = 0;
  S.sc.imu_factor = e->cfg.imu_factor; S.sc.point_distance_factor = e->cfg.point_distance_factor;
  S.sc.prior_factor = e->cfg.prior_factor; S.sc.marginalization_factor = e->cfg.marginalization_factor;
  S.sc.ex_free = e->ex_constant ? 0 : 1;
  S.sc.prior_valid = (e->cfg.marginalization_factor && e->prior.valid) ? 1 : 0;
  S.sc.convergence_flag = e->convergence_flag ? 1 : 0;
  S.sc.turn_off = 1; S.sc.done = 0; S.sc.iteration = 0; S.sc.successful = 0; S.sc.evaluations = 0; S.sc.termination = 0; S.sc.reuse = 0; S.sc.invalid = 0;
  for (int k = 0; k <= O; ++k) { std::memcpy(S.x + 16 * k, e->para_pose[k].data(), 7 * sizeof(double)); std::memcpy(S.x + 16 * k + 7, e->para_sb[k].data(), 9 * sizeof(double)); }
  std::memcpy(S.x + 16 * (O + 1), e->para_ex, 7 * sizeof(double));
  {
    const Tw tt = tlb_double(e);
    S.sc.ex0_pos[0] = tt.pos.x; S.sc.ex0_pos[1] = tt.pos.y; S.sc.ex0_pos[2] = tt.pos.z;
    S.sc.ex0_quat[0] = tt.rot.x; S.sc.ex0_quat[1] = tt.rot.y; S.sc.ex0_quat[2] = tt.rot.z; S.sc.ex0_quat[3] = tt.rot.w;
  }
  for (int i = 0; i < O; ++i) {
    Preintegration &pim = *e->pre[pivot + i + 1];
    S.pim_valid[i] = pim.sum_dt > 10.0 ? 0 : 1;
    S.pim[i] = pim.data();
  }
  if (S.sc.prior_valid) {
    const MargPrior &pr = e->prior;
    std::memcpy(S.bp, pr.bp.data(), sizeof(double) * pr.n);
    S.c0 = pr.c0;
    std::memcpy(S.x0_pose, pr.x0_pose.data(), sizeof(double) * 7 * O);
    std::memcpy(S.x0_sb, pr.x0_sb.data(), sizeof(double) * 9 * O);
    std::memcpy(S.x0_ex, pr.x0_ex, sizeof(double) * 7);
    if (!e->prior_uploaded) {
      EST_CUDA(cudaMemcpyAsync(e->ds.Hp, pr.Hp.d.data(), sizeof(double) * pr.n * pr.n, cudaMemcpyHostToDevice, st));
      e->prior_uploaded = true;
    }
  }
  EST_CUDA(cudaMemcpyAsync(e->ds.st, &S, sizeof(DevSolveState), cudaMemcpyHostToDevice, st));
  for (int i = 1; i <= O; ++i) {
    double Mtmp[108];   // frame terms of the initial point; the solver writes the candidates' terms itself
    ppp_frame_terms(e->para_pose[0].data(), e->para_pose[i].data(), e->para_ex, e->h_Rt + (i - 1) * kAsmRtStride,
                    e->h_Rt + (i - 1) * kAsmRtStride + 9, Mtmp);
  }
  EST_CUDA(cudaMemcpyAsync(e->d_Rt, e->h_Rt, sizeof(double) * O * kAsmRtStride, cudaMemcpyHostToDevice, st));
  e->ds_prepared = true; e->ds_prepared_it = max_it; e->ds_prepared_asm = assemble_only;
  return LIO_OK;
}

static int solve_dev(lio_est *e, int max_it, bool assemble_only) {
  const int O = e->O, pivot = e->W - O;
  cudaStream_t st = e->stream;
  int rc = LIO_OK;
  const double t0 = now_s();
  if (!(e->ds_prepared && e->ds_prepared_it == max_it && e->ds_prepared_asm == assemble_only)) {
    rc = solve_dev_prepare(e, max_it, assemble_only);
    if (rc != LIO_OK) return rc;
  }
  e->ds_prepared = false;
  DevSolveState &S = *e->ds.h_st;
  AsmParams ap;
  std::memset(&ap, 0, sizeof(ap));
  ap.nframes = O;
  long long nfeat = 0;
  for (int i = 1; i <= O; ++i) {
    AsmFrame &f = ap.f[i - 1];
    const FeatureOut &fo = e->feats[pivot + i];
    f.pts = fo.pts; f.coef = fo.coef;
    f.n = (e->cfg.point_distance_factor && (e->fpeers || owns_frame(e, pivot + i))) ? e->h_feat_n[pivot + i] : 0;
    nfeat += f.n;
  }
  asm_plan(ap, e->sm_count);
  ap.skip_flag = &e->ds.st->sc.done;
  ap.stamps = &e->ds.st->dbg[12][0];   // rows 12..14 of the trace: asm_ppp entry / exit stamps per evaluation
  const bool peers = solve_world(e) > 1 && e->npeers == e->world;
  if (solve_world(e) > 1 && !peers && !e->allreduce) {
    lio_set_last_error(__FILE__, __LINE__, "sharded context without an exchange: call lio_est_set_peers or pass an allreduce callback");
    return LIO_ERR_INVALID;
  }
  if (peers) {
    ap.npeers = e->npeers; ap.self = e->rank;
    for (int i = 1; i <= O; ++i) if (owns_frame(e, pivot + i)) ap.owned_mask |= 1u << (i - 1);
  }
  const int nevals = (assemble_only ? 0 : max_it) + 1;
  auto enqueue = [&](cudaStream_t q, bool capturing) -> int {
    // timing events inside a capture must be EXTERNAL event nodes to stay usable with cudaEventElapsedTime
    const unsigned evflag = capturing ? cudaEventRecordExternal : cudaEventRecordDefault;
    for (int ev = 0; ev < nevals; ++ev) {
      int r2 = dev_solver_factors(e->ds, ev, q, &e->launches);   // ImuFactors / prior / M_i on the second stream, beside asm_ppp
      if (r2 != LIO_OK) return r2;
      const double *result = e->asmw.out;
      if (peers) {
        ap.epoch = ++e->xepoch;
        const size_t par = (size_t)(ap.epoch & 1u) * kXRowBytes;
        for (int r = 0; r < e->npeers; ++r) {
          ap.peer_out[r] = reinterpret_cast<double *>(e->peer_base[r] + par);
          ap.peer_flag[r] = reinterpret_cast<unsigned *>(e->peer_base[r] + kXFlagOff);
        }
        result = reinterpret_cast<const double *>(e->xbuf + par);
      }
      // asm_ppp is timed on the first evaluation only: inside the captured graph every event record is a node on the critical path
      // between two k_step launches (measured: the launch behind it starts ~4 us later)
      const bool timed = ev == 0 || (!capturing && solve_world(e) == 1);   // sharded runs: first evaluation only, like the graph
      if (timed) cudaEventRecordWithFlags(e->evp[2 * ev], q, evflag);
      r2 = asm_launch(ap, e->d_Rt, e->asmw, q, &e->launches);
      if (r2 != LIO_OK) return r2;
      if (timed) cudaEventRecordWithFlags(e->evp[2 * ev + 1], q, evflag);
      if (peers) {
        k_xwait<<<1, 32, 0, q>>>(reinterpret_cast<const unsigned *>(e->xbuf + kXFlagOff), e->npeers, ap.epoch,
                                 reinterpret_cast<int *>(e->xbuf + kXErrOff), &e->ds.st->sc.done);
        ++e->launches;
      } else if (solve_world(e) > 1 && e->allreduce) {
        if (e->allreduce(e->allreduce_user, e->asmw.out, O * kAsmStride) != 0) { lio_set_last_error(__FILE__, __LINE__, "allreduce callback failed"); return LIO_ERR_CUDA; }
      }
      r2 = dev_solver_step(e->ds, result, e->d_Rt, ev, q, &e->launches);
      if (r2 != LIO_OK) return r2;
    }
    return LIO_OK;
  };
  if (e->gstream && solve_world(e) == 1 && !assemble_only && max_it == e->cfg.max_num_iterations) {
    // One graph per solve: the launch sequence (and the fork / join with the factor stream) is captured the first time and
    // replayed afterwards; only the asm_ppp nodes are re-parameterised with this scan's feature counts and tile plan.
    cudaStream_t gs = e->gstream;
    EST_CUDA(cudaEventRecord(e->ev_gin, st));
    EST_CUDA(cudaStreamWaitEvent(gs, e->ev_gin, 0));
    if (!e->sexec) {
      asm_prepare();
      const int l0 = e->launches;
      EST_CUDA(cudaStreamBeginCapture(gs, cudaStreamCaptureModeThreadLocal));
      rc = enqueue(gs, true);
      cudaGraph_t g = nullptr;
      const cudaError_t ce = cudaStreamEndCapture(gs, &g);
      if (rc != LIO_OK) { if (g) cudaGraphDestroy(g); return rc; }
      if (ce != cudaSuccess || !g) { lio_set_last_error(__FILE__, __LINE__, cudaGetErrorString(ce)); return LIO_ERR_CUDA; }
      e->sgraph = g;
      e->graph_launches = e->launches - l0;
      e->launches = l0;
      EST_CUDA(cudaGraphInstantiate(&e->sexec, g, 0));
      size_t nn = 0;
      EST_CUDA(cudaGraphGetNodes(g, nullptr, &nn));
      std::vector<cudaGraphNode_t> nodes(nn);
      EST_CUDA(cudaGraphGetNodes(g, nodes.data(), &nn));
      e->asm_nodes.clear();
      for (cudaGraphNode_t nd : nodes) if (asm_is_graph_node(nd)) e->asm_nodes.push_back(nd);
      if ((int)e->asm_nodes.size() != nevals) { lio_set_last_error(__FILE__, __LINE__, "solver graph: unexpected node count"); return LIO_ERR_CUDA; }
    }
    const double tu0 = now_s();
    for (cudaGraphNode_t nd : e->asm_nodes) {
      rc = asm_graph_update(e->sexec, nd, ap, e->d_Rt, e->asmw);
      if (rc != LIO_OK) return rc;
    }
    e->t_lin_lidar = now_s() - tu0;   // device-solver mode: host time of re-parameterising the asm_ppp nodes
    EST_CUDA(cudaGraphLaunch(e->sexec, gs));
    e->t_lin_host = now_s() - t0;     // device-solver mode: host time from the start of the solve to the end of the graph launch call
    e->launches += e->graph_launches;
    EST_CUDA(cudaEventRecord(e->ev_gout, gs));
    EST_CUDA(cudaStreamWaitEvent(st, e->ev_gout, 0));
  } else {
    rc = enqueue(st, false);
    if (rc != LIO_OK) return rc;
  }
  if (peers) EST_CUDA(cudaMemcpyAsync(e->h_S + kMaxOpt * kAsmStride, e->xbuf + kXErrOff, sizeof(int), cudaMemcpyDeviceToHost, st));
  EST_CUDA(cudaMemcpyAsync(&S, e->ds.st, offsetof(DevSolveState, scale), cudaMemcpyDeviceToHost, st));
  EST_CUDA(cudaStreamSynchronize(st));
  if (peers && *reinterpret_cast<const int *>(e->h_S + kMaxOpt * kAsmStride)) {
    cudaMemsetAsync(e->xbuf + kXErrOff, 0, sizeof(int), st);
    *reinterpret_cast<int *>(e->h_S + kMaxOpt * kAsmStride) = 0;
    lio_set_last_error(__FILE__, __LINE__, "peer exchange timed out (a rank did not publish its rows)");
    return LIO_ERR_CUDA;
  }
  const bool graph_replayed = e->sexec && e->gstream && solve_world(e) == 1 && !assemble_only && max_it == e->cfg.max_num_iterations;
  for (int ev = 0; ev < std::min((graph_replayed || solve_world(e) > 1) ? 1 : nevals, S.sc.evaluations); ++ev) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->evp[2 * ev], e->evp[2 * ev + 1]) == cudaSuccess) { e->asm_ms_sum += ms; e->asm_launch_count += 1; e->asm_feat_sum += nfeat; }
    else (void)cudaGetLastError();   // a failed timing query must not surface as the next launch's error
  }
  e->have_H0 = true; e->H0 = Mat(); e->cost0 = S.sc.initial_cost;
  if (assemble_only) return LIO_OK;
  for (int k = 0; k <= O; ++k) { std::memcpy(e->para_pose[k].data(), S.x + 16 * k, 7 * sizeof(double)); std::memcpy(e->para_sb[k].data(), S.x + 16 * k + 7, 9 * sizeof(double)); }
  std::memcpy(e->para_ex, S.x + 16 * (O + 1), 7 * sizeof(double));
  e->S_valid = false;
  e->summary = DoglegSummary();
  e->summary.iterations = S.sc.iteration; e->summary.successful_steps = S.sc.successful; e->summary.evaluations = S.sc.evaluations;
  e->summary.termination = S.sc.termination; e->summary.initial_cost = S.sc.initial_cost; e->summary.final_cost = S.sc.x_cost;
  e->cost_pim = S.sc.cost_pim; e->cost_ppp = S.sc.cost_ppp; e->cost_marg = S.sc.cost_marg;
  e->turn_off = S.sc.turn_off != 0;
  e->convergence_flag = S.sc.convergence_flag != 0;
  e->ex_constant = S.sc.ex_free == 0;
  if (!S.sc.prior_valid) e->prior.valid = false;
  if (S.sc.termination == 2 && !std::isfinite(S.sc.x_cost)) { lio_set_last_error(__FILE__, __LINE__, "solver breakdown"); return LIO_ERR_NUMERIC; }
  e->t_solve = now_s() - t0;
  return LIO_OK;
}

static int scan_solve(lio_est *e, int max_it) { return e->use_dev_solver ? solve_dev(e, max_it, false) : solve_host(e, max_it); }

static int slide_window(lio_est *e) {  // Estimator.cc:2570-2666
  const int W = e->W, O = e->O, pivot = W - O;
  if (e->init_local_map && pivot > 0) {
    const Tw tlb = tlb_double(e);
    const Tw transform_pivot = lidar_pose(e->Ps[pivot], e->Rs[pivot], tlb);
    const int i = pivot + 1;
    const Tw transform_li = lidar_pose(e->Ps[i], e->Rs[i], tlb);
    AffineF a = to_affine_f(tw_mul(tw_inverse(transform_li), transform_pivot));
    ConcatParams cp;
    std::memset(&cp, 0, sizeof(cp));
    cp.nsrc = 2;
    cp.src[0] = e->slot_ptr[e->slot_of[pivot]]; cp.n[0] = e->d_slot_n + e->slot_of[pivot];
    std::memcpy(cp.R[0], a.R, sizeof(a.R)); std::memcpy(cp.t[0], a.t, sizeof(a.t));
    cp.tag[0] = -1.f;
    cp.skip_first[0] = 1; cp.skip_n[0] = e->d_own_n + e->slot_of[0];  // size_surf_stack_[0]
    cp.src[1] = e->slot_ptr[e->slot_of[i]]; cp.n[1] = e->d_slot_n + e->slot_of[i];
    cp.identity[1] = 1;
    k_concat<<<std::max(1, std::min(e->sm_count * 2, (e->slot_cap + 255) / 256)), 256, 0, e->stream>>>(cp, e->d_tmp, e->d_counts + 3, e->slot_cap);
    ++e->launches;
    std::swap(e->slot_ptr[e->slot_of[i]], e->d_tmp);
    EST_CUDA(cudaMemcpyAsync(e->d_slot_n + e->slot_of[i], e->d_counts + 3, sizeof(int), cudaMemcpyDeviceToDevice, e->stream));
  }
  push_shift(e->Ps, e->Ps[W]); push_shift(e->Vs, e->Vs[W]); push_shift(e->Rs, e->Rs[W]); push_shift(e->Bas, e->Bas[W]); push_shift(e->Bgs, e->Bgs[W]);
  return LIO_OK;
}

static int process_scan_body(lio_est *e, const float4 *scan_dev, const int *n_dev, int n_max, bool open_only);
// The pre-integration buffer, the slot rotation and size_surf_stack advance before the fallible device work.  A failure
// after that point leaves the window half-slid, so the context is poisoned: later calls return LIO_ERR_INVALID instead of
// running on inconsistent state (documented in lio_b200.h).
static int process_scan_common(lio_est *e, const float4 *scan_dev, const int *n_dev, int n_max, bool open_only = false) {
  if (e->window_open) { lio_set_last_error(__FILE__, __LINE__, "a scan is open: finish it with lio_est_close_scan first"); return LIO_ERR_INVALID; }
  if (e->poisoned) {
    lio_set_last_error(__FILE__, __LINE__, "estimator context poisoned by an earlier failed scan: destroy and re-create it");
    return LIO_ERR_INVALID;
  }
  if (!e->tmp_pre) { lio_set_last_error(__FILE__, __LINE__, "process_scan before finish_init"); return LIO_ERR_INVALID; }
  const int rc = process_scan_body(e, scan_dev, n_dev, n_max, open_only);
  if (rc != LIO_OK) { e->poisoned = true; std::snprintf(e->err, sizeof(e->err), "%s", lio_last_error()); }
  return rc;
}

static int process_scan_body(lio_est *e, const float4 *scan_dev, const int *n_dev, int n_max, bool open_only) {
  const int W = e->W;
  cudaStream_t st = e->stream;
  marg_start(e);
  const double t0 = now_s();
  e->launches = 0;
  e->t_lin_wait = e->t_lin_host = e->t_lin_lidar = e->t_marg_wait = 0;
  e->have_H0 = false;
  if (!e->tmp_pre) { lio_set_last_error(__FILE__, __LINE__, "process_scan before finish_init"); return LIO_ERR_INVALID; }
  push_shift(e->pre, e->tmp_pre);
  e->tmp_pre = std::make_shared<Preintegration>(e->acc_last, e->gyr_last, e->Bas[W], e->Bgs[W], e->noise);
  // frame slot rotation (CircularBuffer push): the dropped logical frame 0 becomes the new frame W
  {
    const int freed = e->slot_of[0];
    e->slot_of.erase(e->slot_of.begin());
    e->slot_of.push_back(freed);
  }
  const int slot = e->slot_of[W];
  const float4 *src = scan_dev;
  if ((e->cfg.enable_deskew || e->cfg.cutoff_deskew) && !e->cfg.cutoff_deskew && !e->imu_stamped.empty()) {
    // transform_es_ from the IMU-propagated poses of the last 0.1 s (:632-664), float Twist algebra on the host
    const ImuStampedF &te = e->imu_stamped.back();
    ImuStampedF ts = te;
    for (int i = (int)e->imu_stamped.size() - 1; i >= 0; --i) {
      ts = e->imu_stamped[i];
      if (te.time - e->imu_stamped[i].time >= 0.1) break;
    }
    auto twf = [](const float *q, const float *p) { return Tw(Q(q[3], q[0], q[1], q[2]), V3(p[0], p[1], p[2])); };
    // evaluated in double and rounded: the float op order of Eigen::Transform<float> is not reproduced (tolerance-checked)
    Tw body_es = tw_mul(tw_inverse(twf(te.q, te.p)), twf(ts.q, ts.p));
    {
      const float s = (float)(0.1 / (te.time - ts.time));
      Q qe = body_es.rot;
      double d = qe.w, absD = std::fabs(d), s0, s1;
      if (absD >= 1.0 - 1.1920929e-7) { s0 = 1.0 - s; s1 = s; }
      else { double th = std::acos(absD), sn = std::sin(th); s0 = std::sin((1.0 - s) * th) / sn; s1 = std::sin(s * th) / sn; }
      if (d < 0) s1 = -s1;
      body_es.rot = Q(s0 + s1 * qe.w, s1 * qe.x, s1 * qe.y, s1 * qe.z);
      body_es.pos = body_es.pos * (double)s;
    }
    const Tw tlb = tlb_double(e);
    const Tw es = tw_mul(tw_mul(tlb, body_es), tw_inverse(tlb));
    TransformF esf{(float)es.rot.x, (float)es.rot.y, (float)es.rot.z, (float)es.rot.w, (float)es.pos.x, (float)es.pos.y, (float)es.pos.z};
    if (scan_dev != e->d_scan) {
      EST_CUDA(cudaMemcpyAsync(e->d_scan, scan_dev, sizeof(float4) * n_max, cudaMemcpyDeviceToDevice, st));
    }
    k_deskew<<<(n_max + 255) / 256, 256, 0, st>>>(e->d_scan, n_dev, esf, 10.f);
    ++e->launches;
    src = e->d_scan;
  }
  int rc = e->vg.run(src, n_dev, n_max, e->cfg.surf_filter_size, e->slot_ptr[slot], e->cfg.max_frame_points, e->d_slot_n + slot, nullptr, st, &e->launches);
  if (rc != LIO_OK) return rc;
  EST_CUDA(cudaMemcpyAsync(e->d_own_n + slot, e->d_slot_n + slot, sizeof(int), cudaMemcpyDeviceToDevice, st));
  push_shift(e->size_surf_stack, 0);
  rc = scan_open_window(e);
  if (rc != LIO_OK || open_only) return rc;
  rc = scan_solve(e, e->cfg.max_num_iterations);
  if (rc != LIO_OK) return rc;
  rc = scan_close_window(e);
  if (rc != LIO_OK) return rc;
  e->t_total = now_s() - t0;
  return LIO_OK;
}

extern "C" int lio_est_begin_scan(lio_est *e) {
  if (!e) return LIO_ERR_INVALID;
  if (e->cfg.overlap_marginalization) marg_start(e);
  return LIO_OK;
}

extern "C" int lio_est_process_scan_host(lio_est *e, const float *surf_last, int n) {
  if (!e || n < 0 || (n > 0 && !surf_last)) return LIO_ERR_INVALID;
  if (n > e->cfg.max_scan_points) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  if (n > 0) LIO_CUDA_OK(cudaMemcpyAsync(e->d_scan, surf_last, sizeof(float4) * n, cudaMemcpyHostToDevice, e->stream));
  e->h_counts[e->W + 8] = n;
  LIO_CUDA_OK(cudaMemcpyAsync(e->d_counts, e->h_counts + e->W + 8, sizeof(int), cudaMemcpyHostToDevice, e->stream));
  return process_scan_common(e, e->d_scan, e->d_counts, n > 0 ? n : 1);
}

extern "C" int lio_est_process_scan_dev(lio_est *e, const float *surf_last_dev, const int *n_dev, int n_max) {
  if (!e || !surf_last_dev || !n_dev || n_max <= 0) return LIO_ERR_INVALID;
  if (n_max > e->cfg.max_scan_points) n_max = e->cfg.max_scan_points;   // the voxel filter clamps *n_dev to n_max on the device
  LIO_CUDA_OK(cudaSetDevice(e->device));
  return process_scan_common(e, reinterpret_cast<const float4 *>(surf_last_dev), n_dev, n_max);
}

// ---- stepwise API: the phases of ProcessLaserOdom / SolveOptimization one by one ----------------------------------------
extern "C" int lio_est_open_scan_host(lio_est *e, const float *surf_last, int n) {
  if (!e || n < 0 || (n > 0 && !surf_last)) return LIO_ERR_INVALID;
  if (n > e->cfg.max_scan_points) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  if (n > 0) LIO_CUDA_OK(cudaMemcpyAsync(e->d_scan, surf_last, sizeof(float4) * n, cudaMemcpyHostToDevice, e->stream));
  e->h_counts[e->W + 8] = n;
  LIO_CUDA_OK(cudaMemcpyAsync(e->d_counts, e->h_counts + e->W + 8, sizeof(int), cudaMemcpyHostToDevice, e->stream));
  return process_scan_common(e, e->d_scan, e->d_counts, n > 0 ? n : 1, true);
}

extern "C" int lio_est_open_scan_dev(lio_est *e, const float *surf_last_dev, const int *n_dev, int n_max) {
  if (!e || !surf_last_dev || !n_dev || n_max <= 0) return LIO_ERR_INVALID;
  if (n_max > e->cfg.max_scan_points) n_max = e->cfg.max_scan_points;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  return process_scan_common(e, reinterpret_cast<const float4 *>(surf_last_dev), n_dev, n_max, true);
}

static int need_open(lio_est *e) {
  int rc = LIO_OK;
  if (e->poisoned) { lio_set_last_error(__FILE__, __LINE__, "estimator context poisoned by an earlier failed scan: destroy and re-create it"); rc = LIO_ERR_INVALID; }
  else if (!e->window_open) { lio_set_last_error(__FILE__, __LINE__, "no open scan: call lio_est_open_scan_host / _dev first"); rc = LIO_ERR_INVALID; }
  if (rc != LIO_OK) std::snprintf(e->err, sizeof(e->err), "%s", lio_last_error());
  return rc;
}

static void load_parameters(lio_est *e, const double *pose, const double *sb, const double *ex) {
  for (int k = 0; k <= e->O; ++k) {
    if (pose) std::memcpy(e->para_pose[k].data(), pose + 7 * k, 7 * sizeof(double));
    if (sb) std::memcpy(e->para_sb[k].data(), sb + 9 * k, 9 * sizeof(double));
  }
  if (ex) std::memcpy(e->para_ex, ex, 7 * sizeof(double));
  e->S_valid = false;
  e->ds_prepared = false;   // the uploaded solver state belongs to the previous parameter values
}
static void store_parameters(const lio_est *e, double *pose, double *sb, double *ex) {
  for (int k = 0; k <= e->O; ++k) {
    if (pose) std::memcpy(pose + 7 * k, e->para_pose[k].data(), 7 * sizeof(double));
    if (sb) std::memcpy(sb + 9 * k, e->para_sb[k].data(), 9 * sizeof(double));
  }
  if (ex) std::memcpy(ex, e->para_ex, 7 * sizeof(double));
}

extern "C" int lio_est_get_parameters(lio_est *e, double *pose, double *speed_bias, double *ex) {
  if (!e) return LIO_ERR_INVALID;
  int rc = need_open(e);
  if (rc != LIO_OK) return rc;
  store_parameters(e, pose, speed_bias, ex);
  return LIO_OK;
}

extern "C" int lio_est_last_normal_equations(lio_est *e, double *H, double *g, double *cost, int *n);

extern "C" int lio_est_assemble(lio_est *e, const double *pose, const double *speed_bias, const double *ex, double *H, double *g,
                                double *cost, int *n) {
  if (!e || !n) return LIO_ERR_INVALID;
  int rc = need_open(e);
  if (rc != LIO_OK) return rc;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  // evaluate at the caller's blocks, then put the estimator's own blocks back
  std::vector<double> kp(7 * (e->O + 1)), ks(9 * (e->O + 1));
  double kx[7];
  store_parameters(e, kp.data(), ks.data(), kx);
  load_parameters(e, pose, speed_bias, ex);
  if (e->use_dev_solver) {
    rc = solve_dev(e, 0, true);
    if (rc == LIO_OK) rc = lio_est_last_normal_equations(e, H, g, cost, n);
  } else {
    Mat Hh;
    Vec gg;
    double c = 0;
    if (!linearize(e, Hh, gg, c, nullptr, nullptr, nullptr)) { lio_set_last_error(__FILE__, __LINE__, "non-finite cost"); rc = LIO_ERR_NUMERIC; }
    else {
      *n = Hh.r;
      if (H) std::memcpy(H, Hh.d.data(), sizeof(double) * Hh.r * Hh.r);
      if (g) std::memcpy(g, gg.data(), sizeof(double) * Hh.r);
      if (cost) *cost = c;
    }
  }
  load_parameters(e, kp.data(), ks.data(), kx);
  return rc;
}

extern "C" int lio_est_solve(lio_est *e, double *pose, double *speed_bias, double *ex, int max_iter, double summary[8]) {
  if (!e || max_iter < 0) return LIO_ERR_INVALID;
  int rc = need_open(e);
  if (rc != LIO_OK) return rc;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  if (e->use_dev_solver && max_iter > 22) return LIO_ERR_INVALID;
  load_parameters(e, pose, speed_bias, ex);
  rc = scan_solve(e, max_iter);
  if (rc != LIO_OK) { e->poisoned = true; std::snprintf(e->err, sizeof(e->err), "%s", lio_last_error()); return rc; }
  store_parameters(e, pose, speed_bias, ex);
  if (summary) {
    summary[0] = e->summary.iterations; summary[1] = e->summary.successful_steps; summary[2] = e->summary.termination;
    summary[3] = e->summary.initial_cost; summary[4] = e->summary.final_cost; summary[5] = e->summary.evaluations;
    summary[6] = e->convergence_flag ? 1 : 0; summary[7] = e->ex_constant ? 1 : 0;
  }
  return LIO_OK;
}

extern "C" int lio_est_close_scan(lio_est *e, const double *pose, const double *speed_bias, const double *ex) {
  if (!e) return LIO_ERR_INVALID;
  int rc = need_open(e);
  if (rc != LIO_OK) return rc;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  load_parameters(e, pose, speed_bias, ex);
  rc = scan_close_window(e);
  if (rc != LIO_OK) { e->poisoned = true; std::snprintf(e->err, sizeof(e->err), "%s", lio_last_error()); }
  return rc;
}

extern "C" int lio_est_frame_owner(int frame_rel, int world) {  // frame_rel in 1..O (relative to the pivot)
  if (world < 1 || frame_rel < 1) return -1;
  return (frame_rel - 1) % world;
}

extern "C" int lio_est_set_shard(lio_est *e, int rank, int world, lio_allreduce_fn fn, void *user) {
  if (!e || world < 1 || rank < 0 || rank >= world) return LIO_ERR_INVALID;
  e->rank = rank; e->world = world; e->allreduce = fn; e->allreduce_user = user;
  e->npeers = 0;
  e->fpeers = false;
  e->worker.spin_us = world > 1 ? std::max(25.0, 400.0 / world) : 400.0;  // N processes share the host: spin less
  return LIO_OK;
}

extern "C" int lio_est_exchange_buffer(lio_est *e, void **dev_ptr, size_t *bytes) {
  if (!e || !dev_ptr) return LIO_ERR_INVALID;
  *dev_ptr = e->xbuf;
  if (bytes) *bytes = kXBytes;
  return LIO_OK;
}

extern "C" int lio_est_set_peers(lio_est *e, int world, void *const *peer_ptrs) {
  if (!e || !peer_ptrs || world != e->world || world < 2 || world > kMaxPeers) return LIO_ERR_INVALID;
  for (int r = 0; r < world; ++r) {
    e->peer_base[r] = r == e->rank ? e->xbuf : static_cast<char *>(peer_ptrs[r]);
    if (!e->peer_base[r]) return LIO_ERR_INVALID;
  }
  e->npeers = world;
  return LIO_OK;
}

extern "C" int lio_est_feature_slab(lio_est *e, void **dev_ptr, size_t *bytes) {
  if (!e || !dev_ptr) return LIO_ERR_INVALID;
  *dev_ptr = e->fslab;
  if (bytes) *bytes = e->fslab_bytes;
  return LIO_OK;
}

extern "C" int lio_est_set_feature_peers(lio_est *e, int world, void *const *peer_slabs) {
  if (!e || !peer_slabs || world != e->world || world < 2 || world > kMaxPeers) return LIO_ERR_INVALID;
  if (e->window_open) { lio_set_last_error(__FILE__, __LINE__, "lio_est_set_feature_peers inside an open scan"); return LIO_ERR_INVALID; }
  for (int r = 0; r < world; ++r) {
    e->fpeer_base[r] = r == e->rank ? e->fslab : static_cast<char *>(peer_slabs[r]);
    if (!e->fpeer_base[r]) return LIO_ERR_INVALID;
  }
  e->fpeers = true;
  e->npeers = 0;
  return LIO_OK;
}

extern "C" int lio_ipc_export(const void *dev_ptr, unsigned char handle[64]) {
  if (!dev_ptr || !handle) return LIO_ERR_INVALID;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
  cudaIpcMemHandle_t h;
  LIO_CUDA_OK(cudaIpcGetMemHandle(&h, const_cast<void *>(dev_ptr)));
  std::memcpy(handle, &h, 64);
  return LIO_OK;
}

extern "C" int lio_ipc_open(const unsigned char handle[64], void **dev_ptr) {
  if (!handle || !dev_ptr) return LIO_ERR_INVALID;
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle, 64);
  LIO_CUDA_OK(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return LIO_OK;
}

extern "C" int lio_ipc_close(void *dev_ptr) {
  if (!dev_ptr) return LIO_OK;
  LIO_CUDA_OK(cudaIpcCloseMemHandle(dev_ptr));
  return LIO_OK;
}

// ---- getters --------------------------------------------------------------------------------------
extern "C" int lio_est_get_states(lio_est *e, double *out) {
  if (!e || !out) return LIO_ERR_INVALID;
  for (int k = 0; k <= e->W; ++k) {
    double *s = out + 16 * k;
    Q q = fromR(e->Rs[k]);
    s[0] = e->Ps[k].x; s[1] = e->Ps[k].y; s[2] = e->Ps[k].z; s[3] = q.x; s[4] = q.y; s[5] = q.z; s[6] = q.w;
    for (int a = 0; a < 3; ++a) { s[7 + a] = e->Vs[k][a]; s[10 + a] = e->Bas[k][a]; s[13 + a] = e->Bgs[k][a]; }
  }
  return LIO_OK;
}

extern "C" int lio_est_summary(lio_est *e, double *o) {
  if (!e || !o) return LIO_ERR_INVALID;
  const bool has_prior = e->prior.valid || e->mjob.stashed || e->mjob.running;  // does not force the pending algebra
  for (int k = 0; k < 32; ++k) o[k] = 0;
  o[0] = e->summary.iterations; o[1] = e->summary.successful_steps; o[2] = e->summary.termination;
  o[3] = e->summary.initial_cost; o[4] = e->summary.final_cost; o[5] = e->cost_pim; o[6] = e->cost_ppp; o[7] = e->cost_marg;
  o[8] = e->turn_off; o[9] = e->convergence_flag; o[10] = e->h_map_n;
  long long nf = 0;
  for (int v : e->h_feat_n) nf += v;
  o[11] = (double)nf; o[12] = e->odom_iters;
  o[13] = e->t_build; o[14] = e->t_feat; o[15] = e->t_solve; o[16] = e->t_marg; o[17] = e->t_total;
  o[18] = has_prior ? 1 : 0; o[19] = e->summary.evaluations; o[20] = e->summary.evaluations; o[21] = e->launches;
  o[22] = e->t_lin_wait; o[23] = e->t_lin_host; o[24] = e->t_lin_lidar; o[25] = e->t_marg_wait;
  return LIO_OK;
}

extern "C" int lio_est_feature_count(lio_est *e, int frame, int *n) {
  if (!e || !n || frame < 0 || frame > e->W) return LIO_ERR_INVALID;
  *n = e->h_feat_n[frame];
  return LIO_OK;
}

extern "C" int lio_est_get_features(lio_est *e, int frame, float *pts4, float *coef4, int32_t *src, int cap) {
  if (!e || frame < 0 || frame > e->W) return LIO_ERR_INVALID;
  const int n = e->h_feat_n[frame];
  if (n > cap) return LIO_ERR_CAPACITY;
  if (n == 0) return LIO_OK;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  const FeatureOut &f = e->feats[frame];
  if (pts4) LIO_CUDA_OK(cudaMemcpyAsync(pts4, f.pts, sizeof(float4) * n, cudaMemcpyDeviceToHost, e->stream));
  if (coef4) LIO_CUDA_OK(cudaMemcpyAsync(coef4, f.coef, sizeof(float4) * n, cudaMemcpyDeviceToHost, e->stream));
  if (src) LIO_CUDA_OK(cudaMemcpyAsync(src, f.src, sizeof(int) * n, cudaMemcpyDeviceToHost, e->stream));
  LIO_CUDA_OK(cudaStreamSynchronize(e->stream));
  return LIO_OK;
}

extern "C" int lio_est_map_size(lio_est *e, int *n) {
  if (!e || !n) return LIO_ERR_INVALID;
  *n = e->h_map_n;
  return LIO_OK;
}
extern "C" int lio_est_get_map(lio_est *e, float *out, int cap) {
  if (!e || !out) return LIO_ERR_INVALID;
  if (e->h_map_n > cap) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  if (e->h_map_n > 0) LIO_CUDA_OK(cudaMemcpyAsync(out, e->d_map, sizeof(float4) * e->h_map_n, cudaMemcpyDeviceToHost, e->stream));
  LIO_CUDA_OK(cudaStreamSynchronize(e->stream));
  return LIO_OK;
}
extern "C" int lio_est_frame_size(lio_est *e, int frame, int *n) {
  if (!e || !n || frame < 0 || frame > e->W) return LIO_ERR_INVALID;
  LIO_CUDA_OK(cudaSetDevice(e->device));
  LIO_CUDA_OK(cudaMemcpyAsync(n, e->d_slot_n + e->slot_of[frame], sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  LIO_CUDA_OK(cudaStreamSynchronize(e->stream));
  return LIO_OK;
}
extern "C" int lio_est_get_frame(lio_est *e, int frame, float *out, int cap) {
  int n = 0;
  int rc = lio_est_frame_size(e, frame, &n);
  if (rc != LIO_OK) return rc;
  if (n > cap) return LIO_ERR_CAPACITY;
  if (n > 0) LIO_CUDA_OK(cudaMemcpyAsync(out, e->slot_ptr[e->slot_of[frame]], sizeof(float4) * n, cudaMemcpyDeviceToHost, e->stream));
  LIO_CUDA_OK(cudaStreamSynchronize(e->stream));
  return LIO_OK;
}
extern "C" int lio_est_get_local_transform(lio_est *e, int frame, float tf7[7]) {
  if (!e || !tf7 || frame < 0 || frame > e->W) return LIO_ERR_INVALID;
  const TransformF &t = e->local_tf[frame];
  tf7[0] = t.qx; tf7[1] = t.qy; tf7[2] = t.qz; tf7[3] = t.qw; tf7[4] = t.px; tf7[5] = t.py; tf7[6] = t.pz;
  return LIO_OK;
}
extern "C" int lio_est_prior_dim(lio_est *e, int *n) {
  if (!e || !n) return LIO_ERR_INVALID;
  prior_join(e);
  *n = e->prior.valid ? e->prior.n : 0;
  return LIO_OK;
}
extern "C" int lio_est_get_prior(lio_est *e, double *Hp, double *bp) {
  if (!e || !Hp || !bp) return LIO_ERR_INVALID;
  prior_join(e);
  if (!e->prior.valid) return LIO_ERR_INVALID;
  std::memcpy(Hp, e->prior.Hp.d.data(), sizeof(double) * e->prior.n * e->prior.n);
  std::memcpy(bp, e->prior.bp.data(), sizeof(double) * e->prior.n);
  return LIO_OK;
}
extern "C" int lio_est_last_normal_equations(lio_est *e, double *H, double *g, double *cost, int *n) {
  if (!e || !n) return LIO_ERR_INVALID;
  if (!e->have_H0) { *n = 0; return LIO_OK; }
  if (e->use_dev_solver) {
    // device layout keeps the 6 extrinsic slots; report the reduced system when the extrinsic was constant
    const int nf = 15 * (e->O + 1) + 6, nr = e->ex_constant ? nf - 6 : nf;
    *n = nr;
    LIO_CUDA_OK(cudaSetDevice(e->device));
    std::vector<double> Hf((size_t)nf * nf), gf(nf);
    LIO_CUDA_OK(cudaMemcpy(Hf.data(), e->ds.H0, sizeof(double) * nf * nf, cudaMemcpyDeviceToHost));
    LIO_CUDA_OK(cudaMemcpy(gf.data(), e->ds.g0, sizeof(double) * nf, cudaMemcpyDeviceToHost));
    if (H) for (int r = 0; r < nr; ++r) std::memcpy(H + (size_t)r * nr, &Hf[(size_t)r * nf], sizeof(double) * nr);
    if (g) std::memcpy(g, gf.data(), sizeof(double) * nr);
    if (cost) *cost = e->cost0;
    return LIO_OK;
  }
  *n = e->H0.r;
  if (H) std::memcpy(H, e->H0.d.data(), sizeof(double) * e->H0.r * e->H0.r);
  if (g) std::memcpy(g, e->g0.data(), sizeof(double) * e->H0.r);
  if (cost) *cost = e->cost0;
  return LIO_OK;
}
extern "C" int lio_est_last_launches(lio_est *e) { return e ? e->launches : 0; }
extern "C" const char *lio_est_last_error(lio_est *e) { return e ? e->err : "null handle"; }

extern "C" int lio_est_solver_trace(lio_est *e, long long *out, int cap) {
  if (!e || !out || cap < 24 * 16 + 4 * 28 + 4) return LIO_ERR_INVALID;
  if (!e->use_dev_solver) { std::memset(out, 0, sizeof(long long) * (24 * 16 + 4 * 28 + 4)); return LIO_OK; }
  LIO_CUDA_OK(cudaSetDevice(e->device));
  LIO_CUDA_OK(cudaMemcpy(out, reinterpret_cast<const char *>(e->ds.st) + offsetof(DevSolveState, dbg), sizeof(long long) * (24 * 16 + 4 * 28 + 4), cudaMemcpyDeviceToHost));
  return LIO_OK;
}

extern "C" int lio_est_kernel_profile(lio_est *e, double out[8], int reset) {
  if (!e || !out) return LIO_ERR_INVALID;
  out[0] = e->asm_ms_sum; out[1] = (double)e->asm_launch_count; out[2] = (double)e->asm_feat_sum; out[3] = 32.0;
  out[4] = e->knn_ms_sum; out[5] = (double)e->knn_launch_count; out[6] = (double)e->knn_query_sum; out[7] = 128.0;
  if (reset) { e->asm_ms_sum = 0; e->asm_launch_count = 0; e->asm_feat_sum = 0; e->knn_ms_sum = 0; e->knn_launch_count = 0; e->knn_query_sum = 0; }
  return LIO_OK;
}

// ---- factor-operator seam ---------------------------------------------------------------------------
extern "C" int lio_ppp_evaluate(const double point[3], const double coeff[4], const double pose_pivot[7], const double pose_i[7],
                                const double pose_ex[7], double *residual, double *J0, double *J1, double *J2) {
  if (!point || !coeff || !pose_pivot || !pose_i || !pose_ex || !residual) return LIO_ERR_INVALID;
  ppp_evaluate_single(point, coeff, pose_pivot, pose_i, pose_ex, residual, J0, J1, J2);
  return LIO_OK;
}

namespace lio {
int ppp_rows_launch(const float4 *pts, const float4 *coef, int n, const double *Rt12_dev, const double *M_dev, double *r_out,
                    double *J_out, cudaStream_t st);
}

extern "C" int lio_ppp_evaluate_batch_host(const float *pts4, const float *coef4, int n, const double pose_pivot[7],
                                           const double pose_i[7], const double pose_ex[7], double *r_out, double *J_out, int device) {
  if (!pts4 || !coef4 || n < 0 || !pose_pivot || !pose_i || !pose_ex || !r_out || !J_out) return LIO_ERR_INVALID;
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  if (n == 0) return LIO_OK;
  LIO_CUDA_OK(cudaSetDevice(device));
  double Rt[12], M[108];
  ppp_frame_terms(pose_pivot, pose_i, pose_ex, Rt, Rt + 9, M);
  float4 *dp = nullptr, *dc = nullptr;
  double *dRt = nullptr, *dM = nullptr, *dr = nullptr, *dJ = nullptr;
  int rc = LIO_OK;
  if (cudaMalloc(&dp, sizeof(float4) * n) != cudaSuccess || cudaMalloc(&dc, sizeof(float4) * n) != cudaSuccess ||
      cudaMalloc(&dRt, sizeof(Rt)) != cudaSuccess || cudaMalloc(&dM, sizeof(M)) != cudaSuccess ||
      cudaMalloc(&dr, sizeof(double) * n) != cudaSuccess || cudaMalloc(&dJ, sizeof(double) * 18 * (size_t)n) != cudaSuccess) {
    lio_set_last_error(__FILE__, __LINE__, "cudaMalloc failed");
    rc = LIO_ERR_CUDA;
  }
  if (rc == LIO_OK) {
    cudaMemcpy(dp, pts4, sizeof(float4) * n, cudaMemcpyHostToDevice);
    cudaMemcpy(dc, coef4, sizeof(float4) * n, cudaMemcpyHostToDevice);
    cudaMemcpy(dRt, Rt, sizeof(Rt), cudaMemcpyHostToDevice);
    cudaMemcpy(dM, M, sizeof(M), cudaMemcpyHostToDevice);
    rc = ppp_rows_launch(dp, dc, n, dRt, dM, dr, dJ, 0);
    if (rc == LIO_OK) {
      cudaError_t er = cudaMemcpy(r_out, dr, sizeof(double) * n, cudaMemcpyDeviceToHost);
      if (er == cudaSuccess) er = cudaMemcpy(J_out, dJ, sizeof(double) * 18 * (size_t)n, cudaMemcpyDeviceToHost);
      if (er != cudaSuccess) { lio_set_last_error(__FILE__, __LINE__, cudaGetErrorString(er)); rc = LIO_ERR_CUDA; }
    }
  }
  void *fr[] = {dp, dc, dRt, dM, dr, dJ};
  for (void *q : fr) if (q) cudaFree(q);
  return rc;
}

// Stage C reduction of ONE frame on explicit host arrays (parity entry for the fused kernel):
// out32[0..27] = upper triangle of S = sum rho'(r^2) [g;r][g;r]^T, out32[28] = sum log(1+r^2).
extern "C" int lio_asm_ppp_host(const float *pts4, const float *coef4, int n, const double R9[9], const double t3[3],
                                double out32[32], int device) {
  if (!pts4 || !coef4 || n < 0 || !R9 || !t3 || !out32) return LIO_ERR_INVALID;
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  LIO_CUDA_OK(cudaSetDevice(device));
  AsmWork w;
  float4 *dp = nullptr, *dc = nullptr;
  int rc = LIO_OK;
  const int nn = n > 0 ? n : 1;
  if (w.init(nn) != 0 || cudaMalloc(&dp, sizeof(float4) * nn) != cudaSuccess || cudaMalloc(&dc, sizeof(float4) * nn) != cudaSuccess) {
    lio_set_last_error(__FILE__, __LINE__, "cudaMalloc failed");
    rc = LIO_ERR_CUDA;
  }
  if (rc == LIO_OK) {
    cudaMemcpy(dp, pts4, sizeof(float4) * n, cudaMemcpyHostToDevice);
    cudaMemcpy(dc, coef4, sizeof(float4) * n, cudaMemcpyHostToDevice);
    AsmParams ap;
    std::memset(&ap, 0, sizeof(ap));
    ap.nframes = 1;
    ap.f[0].pts = dp; ap.f[0].coef = dc; ap.f[0].n = n;
    double Rt[kAsmRtStride];
    std::memcpy(Rt, R9, sizeof(double) * 9); std::memcpy(Rt + 9, t3, sizeof(double) * 3);
    double *dRt = nullptr;
    cudaMalloc(&dRt, sizeof(Rt));
    cudaMemcpy(dRt, Rt, sizeof(Rt), cudaMemcpyHostToDevice);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    asm_plan(ap, sms);
    rc = asm_launch(ap, dRt, w, 0, nullptr);
    cudaDeviceSynchronize();
    cudaFree(dRt);
    if (rc == LIO_OK) {
      cudaError_t er = cudaMemcpy(out32, w.out, sizeof(double) * kAsmStride, cudaMemcpyDeviceToHost);
      if (er != cudaSuccess) { lio_set_last_error(__FILE__, __LINE__, cudaGetErrorString(er)); rc = LIO_ERR_CUDA; }
    }
  }
  if (dp) cudaFree(dp);
  if (dc) cudaFree(dc);
  w.destroy();
  return rc;
}

// Synthetic feature stream shaped like a converged window: points within +-20 m, unit normals scaled by a score of 0.8,
// and plane offsets chosen so that the residual under the frame's (R, t) of the benchmark is a few centimetres
// (|r| <= 0.04 m), i.e. the regime the solver runs in (rho = log(1 + r^2) with r^2 << 1).
__global__ void k_fill_features(float4 *pts, float4 *coef, long long n, long long per_frame) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned h = (unsigned)(i * 2654435761u);
  float a = (float)(h & 1023) * (1.0f / 1024.0f), b = (float)((h >> 10) & 1023) * (1.0f / 1024.0f), c = (float)((h >> 20) & 1023) * (1.0f / 1024.0f);
  const float px = 40.f * (a - 0.5f), py = 40.f * (b - 0.5f), pz = 4.f * c;
  pts[i] = make_float4(px, py, pz, 0.9f);
  float nx = a - 0.5f, ny = b - 0.5f, nz = c + 0.1f, nn = rsqrtf(nx * nx + ny * ny + nz * nz);
  const float wx = 0.8f * nx * nn, wy = 0.8f * ny * nn, wz = 0.8f * nz * nn;
  // same (R, t) as lio_asm_stream_bench builds for frame k: R = Rz(0.01 k) stored row-major, t = (0.1 k, 0.02 k, 0)
  const int k = (int)(i / per_frame);
  const double cs = cos(0.01 * k), sn = sin(0.01 * k);
  const double ax = cs * wx + sn * wy, ay = -sn * wx + cs * wy, az = wz;   // a = R^T w
  const double r0 = ax * (px + 0.1 * k) + ay * (py + 0.02 * k) + az * pz;
  coef[i] = make_float4(wx, wy, wz, (float)(-r0) + 0.08f * (a - 0.5f));
}

// Streaming-rate measurement of the fused stage-C kernel on a synthetic feature stream of n features
// (choose n*32 B larger than L2 to measure the HBM-resident rate).  CUDA events around each launch on the
// launching stream.  out = {avg ms per launch, min ms, bytes per launch, launches}.
// ---- C-ABI: TransformToEnd on an explicit host array (parity entry) ----------------------------------------------
extern "C" int lio_transform_to_end_host(float *cloud, int n, const float *tf7_es, float time_factor, int device) {
  if (!cloud || !tf7_es || n < 0) return LIO_ERR_INVALID;
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  LIO_CUDA_OK(cudaSetDevice(device));
  if (n == 0) return LIO_OK;
  float4 *d = nullptr;
  int *dn = nullptr;
  LIO_CUDA_OK(cudaMalloc(&d, sizeof(float4) * n));
  cudaError_t ce = cudaMalloc(&dn, sizeof(int));
  if (ce == cudaSuccess) ce = cudaMemcpy(d, cloud, sizeof(float4) * n, cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(dn, &n, sizeof(int), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) {
    TransformF es;
    std::memcpy(&es, tf7_es, sizeof(es));
    k_deskew<<<(n + 255) / 256, 256>>>(d, dn, es, time_factor);
    ce = cudaMemcpy(cloud, d, sizeof(float4) * n, cudaMemcpyDeviceToHost);
  }
  cudaFree(d);
  if (dn) cudaFree(dn);
  if (ce != cudaSuccess) { lio_set_last_error(__FILE__, __LINE__, cudaGetErrorString(ce)); return LIO_ERR_CUDA; }
  return LIO_OK;
}

// ---- PointMapping::OptimizeTransformTobeMapped (PointMapping.cc:325-753) on device-resident clouds -----------------------
namespace lio {

int ScanToMapWork::init(int cap_corner_map, int cap_surf_map, int cap_queries) {
  cap_feat = cap_queries > 0 ? cap_queries : 1;
  if (hc.init(cap_corner_map > 0 ? cap_corner_map : 1) != 0 || hs.init(cap_surf_map > 0 ? cap_surf_map : 1) != 0 || w.init(cap_feat + 1) != 0) return -1;
  auto alloc = [](void **p, size_t bytes) { return cudaMalloc(p, bytes ? bytes : 16) == cudaSuccess; };
  if (!(alloc((void **)&fo.pts, sizeof(float4) * cap_feat) && alloc((void **)&fo.coef, sizeof(float4) * cap_feat) &&
        alloc((void **)&fo.src, sizeof(int) * cap_feat) && alloc((void **)&d_n, sizeof(int) * 8) && alloc((void **)&d_tf, sizeof(TransformF)) &&
        alloc((void **)&d_odom, sizeof(OdomState)) && alloc((void **)&d_partial, sizeof(double) * 32 * 1024) && alloc((void **)&d_z, sizeof(float) * 4) &&
        cudaMallocHost((void **)&h_stage, 64) == cudaSuccess))
    return -1;
  fo.cap = cap_feat;
  fo.count = d_n + 4;
  return 0;
}

void ScanToMapWork::destroy() {
  void *fr[] = {fo.pts, fo.coef, fo.src, d_n, d_tf, d_odom, d_partial, d_z};
  for (void *q : fr) if (q) cudaFree(q);
  if (h_stage) cudaFreeHost(h_stage);
  hc.destroy(); hs.destroy(); w.destroy();
  fo = FeatureOut(); d_n = nullptr; d_tf = nullptr; d_odom = nullptr; d_partial = nullptr; d_z = nullptr; h_stage = nullptr;
}

// Maps and stacks are device arrays; Kc / Ks are known on the host (the caller assembled the maps), the stack sizes are
// device counts bounded by Mc_max / Ms_max.  tf7 (host, in/out).  The uploads go through the workspace's pinned staging,
// so the only synchronisation is the final read-back.  stats (optional) accumulates launches, the sync and the copies.
int scan_to_map_run(ScanToMapWork &W, const float4 *d_cmap, int Kc, const float4 *d_smap, int Ks, const float4 *d_corner, const int *d_nc,
                    int Mc_max, const float4 *d_surf, const int *d_ns, int Ms_max, float *tf7, float min_match_sq_dis, float min_plane_dis,
                    int max_iter, double delta_r_abort, double delta_t_abort, int variant, int *n_out, int *iters, int sm, cudaStream_t st,
                    CallStats *stats) {
  if (n_out) *n_out = 0;
  if (iters) *iters = 0;
  if (Kc <= 10 || Ks <= 100 || max_iter == 0) return LIO_OK;  // PointMapping.cc:327-329: nothing to optimise against
  if (Mc_max + Ms_max > W.cap_feat) { lio_set_last_error(__FILE__, __LINE__, "scan-to-map: stacks exceed the feature capacity"); return LIO_ERR_CAPACITY; }
  CallStats local;
  CallStats &S = stats ? *stats : local;
  int *hn = reinterpret_cast<int *>(W.h_stage);              // [0, 8)   Kc, Ks
  float *hz = reinterpret_cast<float *>(W.h_stage + 16);     // [16, 32) point_on_z_axis_
  float *htf = reinterpret_cast<float *>(W.h_stage + 32);    // [32, 60) start pose
  hn[0] = Kc; hn[1] = Ks;
  std::memcpy(htf, tf7, sizeof(TransformF));
  LIO_CUDA_OK(stats_h2d(S, W.d_n, hn, 2 * sizeof(int), st));
  LIO_CUDA_OK(cudaMemsetAsync(W.d_n + 4, 0, sizeof(int), st));
  LIO_CUDA_OK(stats_h2d(S, W.d_tf, htf, sizeof(TransformF), st));
  LIO_CUDA_OK(cudaMemsetAsync(W.d_odom, 0, sizeof(OdomState), st));
  {  // point_on_z_axis_ = T0 * (0, 0, 10), fixed for the whole optimisation (PointMapping.cc:803-806); float, no FMA
    const float qx = tf7[0], qy = tf7[1], qz = tf7[2], qw = tf7[3], vx = 0.0f, vy = 0.0f, vz = 10.0f;
    volatile float ux = qy * vz - qz * vy, uy = qz * vx - qx * vz, uz = qx * vy - qy * vx;
    volatile float ux2 = ux + ux, uy2 = uy + uy, uz2 = uz + uz;
    volatile float cx = qy * uz2 - qz * uy2, cy = qz * ux2 - qx * uz2, cz = qx * uy2 - qy * ux2;
    volatile float ax = ux2 * qw, ay = uy2 * qw, az = uz2 * qw;
    volatile float rx = vx + ax, ry = vy + ay, rz = vz + az;
    volatile float sx = rx + cx, sy = ry + cy, sz = rz + cz;
    hz[0] = sx + tf7[4]; hz[1] = sy + tf7[5]; hz[2] = sz + tf7[6]; hz[3] = 0.f;
    LIO_CUDA_OK(stats_h2d(S, W.d_z, hz, 4 * sizeof(float), st));
  }
  const float cell = sqrtf(min_match_sq_dis) * (1.0f + 1.0f / 1024.0f);
  int launches = 0;
  int rc = W.hc.build(d_cmap, W.d_n, Kc, cell, st, &launches);
  if (rc == LIO_OK) rc = W.hs.build(d_smap, W.d_n + 1, Ks, cell, st, &launches);
  const int cap = std::max(1, Mc_max + Ms_max);
  const int nb = std::max(1, std::min(sm, (cap + kOdomThreads - 1) / kOdomThreads));
  for (int it = 0; it < max_iter && rc == LIO_OK; ++it) {
    rc = calculate_features_dev(W.hc, d_cmap, d_corner, d_nc, std::max(Mc_max, 1), W.d_tf, min_match_sq_dis, min_plane_dis, W.fo, 0,
                                &W.d_odom->done, W.w, st, &launches, 3, W.d_z);
    if (rc == LIO_OK)
      rc = calculate_features_dev(W.hs, d_smap, d_surf, d_ns, std::max(Ms_max, 1), W.d_tf, min_match_sq_dis, min_plane_dis, W.fo, 1,
                                  &W.d_odom->done, W.w, st, &launches, 2, W.d_z);
    if (rc != LIO_OK) break;
    k_odom_reduce<<<nb, kOdomThreads, 0, st>>>(W.fo.pts, W.fo.coef, W.fo.count, W.d_tf, W.d_odom, W.d_partial, variant == 1 ? 2 : 1);
    k_odom_solve<<<1, 32, 0, st>>>(W.d_odom, W.d_tf, delta_r_abort, delta_t_abort, it, W.fo.count, 50, variant == 1 ? 1 : 0);
    launches += 2;
  }
  S.launches += launches;
  if (rc != LIO_OK) return rc;
  int m = 0, it_done = 0;
  cudaError_t ce = stats_d2h(S, &m, W.d_n + 4, sizeof(int), st);
  if (ce == cudaSuccess) ce = stats_d2h(S, &it_done, &W.d_odom->iter, sizeof(int), st);
  if (ce == cudaSuccess) ce = stats_d2h(S, tf7, W.d_tf, sizeof(TransformF), st);
  if (ce == cudaSuccess) ce = stats_sync(S, st);
  if (ce != cudaSuccess) { lio_set_last_error(__FILE__, __LINE__, cudaGetErrorString(ce)); return LIO_ERR_CUDA; }
  if (m > cap) { lio_set_last_error(__FILE__, __LINE__, "feature buffer overflow"); return LIO_ERR_CAPACITY; }
  if (n_out) *n_out = m;
  if (iters) *iters = it_done;
  return LIO_OK;
}

}  // namespace lio

// ---- C-ABI: PointMapping::OptimizeTransformTobeMapped on explicit host arrays (parity entry) ------------------------
extern "C" int lio_scan_to_map_host(const float *corner_map, int Kc, const float *surf_map, int Ks, const float *corner, int Mc,
                                    const float *surf, int Ms, float *tf7, float min_match_sq_dis, float min_plane_dis, int max_iter,
                                    double delta_r_abort, double delta_t_abort, int variant, float *pts4, float *coef4, int32_t *src,
                                    int *n_out, int *iters, int device) {
  if (!corner_map || !surf_map || !corner || !surf || !tf7 || Kc < 0 || Ks < 0 || Mc < 0 || Ms < 0 || max_iter < 0 || variant < 0 || variant > 1)
    return LIO_ERR_INVALID;
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  LIO_CUDA_OK(cudaSetDevice(device));
  if (n_out) *n_out = 0;
  if (iters) *iters = 0;
  if (Kc <= 10 || Ks <= 100 || max_iter == 0) return LIO_OK;  // PointMapping.cc:327-329: nothing to optimise against
  ScanToMapWork W;
  float4 *d_cmap = nullptr, *d_smap = nullptr, *d_corner = nullptr, *d_surf = nullptr;
  int *d_cnt = nullptr;
  int rc = LIO_OK, sm = 148;
  cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device);
  auto alloc = [&](void **p, size_t bytes) { return cudaMalloc(p, bytes ? bytes : 16) == cudaSuccess; };
  if (W.init(Kc, Ks, Mc + Ms) != 0 || !(alloc((void **)&d_cmap, sizeof(float4) * Kc) && alloc((void **)&d_smap, sizeof(float4) * Ks) &&
                                         alloc((void **)&d_corner, sizeof(float4) * Mc) && alloc((void **)&d_surf, sizeof(float4) * Ms) &&
                                         alloc((void **)&d_cnt, sizeof(int) * 2))) {
    lio_set_last_error(__FILE__, __LINE__, "cudaMalloc failed");
    rc = LIO_ERR_CUDA;
  }
  if (rc == LIO_OK) {
    const int hn[2] = {Mc, Ms};
    cudaMemcpy(d_cmap, corner_map, sizeof(float4) * Kc, cudaMemcpyHostToDevice);
    cudaMemcpy(d_smap, surf_map, sizeof(float4) * Ks, cudaMemcpyHostToDevice);
    if (Mc) cudaMemcpy(d_corner, corner, sizeof(float4) * Mc, cudaMemcpyHostToDevice);
    if (Ms) cudaMemcpy(d_surf, surf, sizeof(float4) * Ms, cudaMemcpyHostToDevice);
    cudaMemcpy(d_cnt, hn, sizeof(hn), cudaMemcpyHostToDevice);
    int m = 0;
    rc = scan_to_map_run(W, d_cmap, Kc, d_smap, Ks, d_corner, d_cnt, Mc, d_surf, d_cnt + 1, Ms, tf7, min_match_sq_dis, min_plane_dis, max_iter,
                         delta_r_abort, delta_t_abort, variant, &m, iters, sm, 0);
    if (rc == LIO_OK) {
      if (n_out) *n_out = m;
      if (m > 0) {
        if (pts4) cudaMemcpy(pts4, W.fo.pts, sizeof(float4) * m, cudaMemcpyDeviceToHost);
        if (coef4) cudaMemcpy(coef4, W.fo.coef, sizeof(float4) * m, cudaMemcpyDeviceToHost);
        if (src) cudaMemcpy(src, W.fo.src, sizeof(int) * m, cudaMemcpyDeviceToHost);
      }
    }
  }
  void *fr[] = {d_cmap, d_smap, d_corner, d_surf, d_cnt};
  for (void *q : fr) if (q) cudaFree(q);
  W.destroy();
  return rc;
}

// ---- C-ABI: Estimator::CalculateLaserOdom on explicit host arrays (parity entry) ---------------------------------
extern "C" int lio_laser_odom_host(const float *map, int K, const float *surf, int M, float *tf7, float min_match_sq_dis,
                                   float min_plane_dis, int keep_features, int max_iter, float *pts4, float *coef4, int32_t *src,
                                   int *n_out, int *iters, int device) {
  if (!map || !surf || !tf7 || !n_out || K < 0 || M < 0 || max_iter < 0) return LIO_ERR_INVALID;
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  LIO_CUDA_OK(cudaSetDevice(device));
  *n_out = 0;
  if (iters) *iters = 0;
  if (M == 0 || max_iter == 0) return LIO_OK;
  const int cap = M * (keep_features ? max_iter : 1);
  CellHash h;
  KnnWork w;
  float4 *d_map = nullptr, *d_surf = nullptr;
  FeatureOut fo;
  int *d_n = nullptr;
  TransformF *d_tf = nullptr;
  OdomState *d_odom = nullptr;
  double *d_partial = nullptr;
  int rc = LIO_OK, sm = 148;
  cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device);
  const int Kc = K > 0 ? K : 1;
  if (h.init(Kc) != 0 || w.init(M) != 0) rc = LIO_ERR_CUDA;
  if (rc == LIO_OK && (cudaMalloc(&d_map, sizeof(float4) * Kc) != cudaSuccess || cudaMalloc(&d_surf, sizeof(float4) * M) != cudaSuccess ||
                       cudaMalloc(&fo.pts, sizeof(float4) * cap) != cudaSuccess || cudaMalloc(&fo.coef, sizeof(float4) * cap) != cudaSuccess ||
                       cudaMalloc(&fo.src, sizeof(int) * cap) != cudaSuccess || cudaMalloc(&d_n, sizeof(int) * 4) != cudaSuccess ||
                       cudaMalloc(&d_tf, sizeof(TransformF)) != cudaSuccess || cudaMalloc(&d_odom, sizeof(OdomState)) != cudaSuccess ||
                       cudaMalloc(&d_partial, sizeof(double) * 32 * 1024) != cudaSuccess))
    rc = LIO_ERR_CUDA;
  if (rc != LIO_OK) lio_set_last_error(__FILE__, __LINE__, "cudaMalloc failed");
  if (rc == LIO_OK) {
    const int hn[3] = {K, M, 0};
    cudaMemcpy(d_map, map, sizeof(float4) * K, cudaMemcpyHostToDevice);
    cudaMemcpy(d_surf, surf, sizeof(float4) * M, cudaMemcpyHostToDevice);
    cudaMemcpy(d_n, hn, sizeof(hn), cudaMemcpyHostToDevice);
    cudaMemcpy(d_tf, tf7, sizeof(TransformF), cudaMemcpyHostToDevice);
    cudaMemset(d_odom, 0, sizeof(OdomState));
    fo.count = d_n + 2; fo.cap = cap;
    const float cell = sqrtf(min_match_sq_dis) * (1.0f + 1.0f / 1024.0f);
    rc = h.build(d_map, d_n, Kc, cell, 0, nullptr);
    const int nb = std::max(1, std::min(sm, (cap + kOdomThreads - 1) / kOdomThreads));
    for (int it = 0; it < max_iter && rc == LIO_OK; ++it) {
      rc = calculate_features_dev(h, d_map, d_surf, d_n + 1, M, d_tf, min_match_sq_dis, min_plane_dis, fo, keep_features ? 1 : 0,
                                  &d_odom->done, w, 0, nullptr);
      if (rc != LIO_OK) break;
      k_odom_reduce<<<nb, kOdomThreads>>>(fo.pts, fo.coef, fo.count, d_tf, d_odom, d_partial);
      k_odom_solve<<<1, 32>>>(d_odom, d_tf, 0.05, 0.05);
    }
    if (rc == LIO_OK) {
      int m = 0;
      OdomState hs;
      cudaError_t ce = cudaMemcpy(&m, d_n + 2, sizeof(int), cudaMemcpyDeviceToHost);
      if (ce == cudaSuccess) ce = cudaMemcpy(&hs, d_odom, sizeof(OdomState), cudaMemcpyDeviceToHost);
      if (ce == cudaSuccess) ce = cudaMemcpy(tf7, d_tf, sizeof(TransformF), cudaMemcpyDeviceToHost);
      if (ce != cudaSuccess) { lio_set_last_error(__FILE__, __LINE__, cudaGetErrorString(ce)); rc = LIO_ERR_CUDA; }
      else if (m > cap) { lio_set_last_error(__FILE__, __LINE__, "feature buffer overflow"); rc = LIO_ERR_CAPACITY; }
      else {
        *n_out = m;
        if (iters) *iters = hs.iter;
        if (m > 0) {
          if (pts4) cudaMemcpy(pts4, fo.pts, sizeof(float4) * m, cudaMemcpyDeviceToHost);
          if (coef4) cudaMemcpy(coef4, fo.coef, sizeof(float4) * m, cudaMemcpyDeviceToHost);
          if (src) cudaMemcpy(src, fo.src, sizeof(int) * m, cudaMemcpyDeviceToHost);
        }
      }
    }
  }
  void *fr[] = {d_map, d_surf, fo.pts, fo.coef, fo.src, d_n, d_tf, d_odom, d_partial};
  for (void *q : fr) if (q) cudaFree(q);
  h.destroy();
  w.destroy();
  return rc;
}

extern "C" int lio_asm_set_fold_chunks(int chunks) {
  asm_set_fold_chunks(chunks);
  return LIO_OK;
}

extern "C" int lio_asm_stream_bench(long long n_features, int iters, int device, double out[4]) {
  if (n_features <= 0 || iters <= 0 || !out) return LIO_ERR_INVALID;
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  LIO_CUDA_OK(cudaSetDevice(device));
  const int O = 8;  // spread over 8 equal frames like a window
  const long long per = n_features / O;
  if (per <= 0 || per > 0x7fffffffLL) return LIO_ERR_INVALID;
  float4 *dp = nullptr, *dc = nullptr;
  AsmWork w;
  int rc = LIO_OK;
  if (cudaMalloc(&dp, sizeof(float4) * per * O) != cudaSuccess || cudaMalloc(&dc, sizeof(float4) * per * O) != cudaSuccess ||
      w.init((int)std::min<long long>(per * O, 1ll << 30)) != 0) {
    lio_set_last_error(__FILE__, __LINE__, "cudaMalloc failed");
    rc = LIO_ERR_CUDA;
  }
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  double *dRt = nullptr;
  if (rc == LIO_OK) {
    k_fill_features<<<(unsigned)((per * O + 255) / 256), 256>>>(dp, dc, per * O, per);
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    AsmParams ap;
    std::memset(&ap, 0, sizeof(ap));
    ap.nframes = O;
    double hRt[8 * kAsmRtStride];
    for (int k = 0; k < O; ++k) {
      ap.f[k].pts = dp + per * k; ap.f[k].coef = dc + per * k; ap.f[k].n = (int)per;
      const double c = std::cos(0.01 * k), s = std::sin(0.01 * k);
      const double Rt[kAsmRtStride] = {c, -s, 0, s, c, 0, 0, 0, 1, 0.1 * k, 0.02 * k, 0.0};
      std::memcpy(hRt + k * kAsmRtStride, Rt, sizeof(Rt));
    }
    cudaMalloc(&dRt, sizeof(hRt));
    cudaMemcpy(dRt, hRt, sizeof(hRt), cudaMemcpyHostToDevice);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    asm_plan(ap, sms);
    double sum = 0, mn = 1e30;
    for (int it = 0; it < iters + 3 && rc == LIO_OK; ++it) {
      cudaEventRecord(e0, 0);
      rc = asm_launch(ap, dRt, w, 0, nullptr);
      cudaEventRecord(e1, 0);
      if (cudaEventSynchronize(e1) != cudaSuccess) { lio_set_last_error(__FILE__, __LINE__, "kernel failed"); rc = LIO_ERR_CUDA; break; }
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      if (it >= 3) { sum += ms; mn = std::min(mn, (double)ms); }
    }
    out[0] = sum / iters; out[1] = mn; out[2] = 32.0 * (double)(per * O); out[3] = iters;
  }
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  if (dRt) cudaFree(dRt);
  if (dp) cudaFree(dp);
  if (dc) cudaFree(dc);
  w.destroy();
  return rc;
}

extern "C" int lio_pim_create(const double a0[3], const double g0[3], const double ba[3], const double bg[3], const double n5[5], lio_pim **out) {
  if (!a0 || !g0 || !ba || !bg || !n5 || !out) return LIO_ERR_INVALID;
  ImuNoise nz;
  nz.acc_n = n5[0]; nz.gyr_n = n5[1]; nz.acc_w = n5[2]; nz.gyr_w = n5[3]; nz.g_norm = n5[4];
  lio_pim *p = new (std::nothrow) lio_pim();
  if (!p) return LIO_ERR_INVALID;
  p->p = std::make_shared<Preintegration>(V3(a0), V3(g0), V3(ba), V3(bg), nz);
  *out = p;
  return LIO_OK;
}
extern "C" int lio_pim_destroy(lio_pim *p) { delete p; return LIO_OK; }
extern "C" int lio_pim_push_back(lio_pim *p, double dt, const double a[3], const double g[3]) {
  if (!p || !a || !g) return LIO_ERR_INVALID;
  p->p->push_back(dt, V3(a), V3(g));
  return LIO_OK;
}
extern "C" int lio_pim_get(lio_pim *p, double *s, double *jac, double *cov) {
  if (!p || !s) return LIO_ERR_INVALID;
  const Preintegration &q = *p->p;
  s[0] = q.delta_p.x; s[1] = q.delta_p.y; s[2] = q.delta_p.z; s[3] = q.delta_q.x; s[4] = q.delta_q.y; s[5] = q.delta_q.z; s[6] = q.delta_q.w;
  s[7] = q.delta_v.x; s[8] = q.delta_v.y; s[9] = q.delta_v.z; s[10] = q.sum_dt;
  if (jac) std::memcpy(jac, q.jac, sizeof(q.jac));
  if (cov) std::memcpy(cov, q.cov, sizeof(q.cov));
  return LIO_OK;
}
extern "C" int lio_imu_factor_evaluate(lio_pim *p, const double pose_i[7], const double sb_i[9], const double pose_j[7],
                                       const double sb_j[9], double *res15, double *J0, double *J1, double *J2, double *J3) {
  if (!p || !pose_i || !sb_i || !pose_j || !sb_j || !res15) return LIO_ERR_INVALID;
  double Ji[15][6], Jsi[15][9], Jj[15][6], Jsj[15][9];
  const bool need = J0 || J1 || J2 || J3;
  imu_factor_evaluate(*p->p, pose_i, sb_i, pose_j, sb_j, res15, need ? Ji : nullptr, Jsi, Jj, Jsj);
  if (need) {
    for (int a = 0; a < 15; ++a) {
      for (int c = 0; c < 7; ++c) { if (J0) J0[a * 7 + c] = c < 6 ? Ji[a][c] : 0.0; if (J2) J2[a * 7 + c] = c < 6 ? Jj[a][c] : 0.0; }
      for (int c = 0; c < 9; ++c) { if (J1) J1[a * 9 + c] = Jsi[a][c]; if (J3) J3[a * 9 + c] = Jsj[a][c]; }
    }
  }
  return LIO_OK;
}

