// lio::PointMapping's rolling cube map and its Process() step (pre-initialisation scan-to-map path) with the map resident in
// HBM - SURVEY section 8 row f2.  Reference: src/point_processor/PointMapping.cc
//   constants / ToIndex        :77-82, :121-122, include/point_processor/PointMapping.h:150-159   (21 x 21 x 11 cubes of 50 m)
//   re-centring                :809-931      cube descriptors are shifted on the host: no point moves in HBM
//   cube selection             :944-1003     5 x 5 x 5 neighbourhood, FOV test on the eight cube corners (host, <= 125 cubes)
//   map extraction             :1005-1011    one gather kernel over the valid cubes' HBM segments
//   Process                    :765-1052     PointAssociateToMap / TobeMapped kernels, VoxelGrid of the stacks,
//                                            OptimizeTransformTobeMapped (scan_to_map_run: voxel-hash k-NN + 6 x 6 float GN)
//   UpdateMapDatabase          :1112-1208    order-preserving insert into the cubes + VoxelGrid of every touched valid cube
// Per-point work runs in kernels; the 4851-entry cube directory (pointer, count, capacity per cube) lives on the host and is
// the only thing the control logic touches.  The insert is a stable radix sort of (cube, input index) followed by a scatter
// to `append position of the cube + rank in its run`; the host reads only the per-cube add counts, grows the segments and
// uploads the append positions of the touched cubes (the device mirror of the directory the scatter reads).  Compiled with -fmad=false: the float expressions follow the reference's order,
// clouds, cube contents and the mapped pose are compared with the oracle (oracle/o_cubemap.cc).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>
#include "odom.cuh"
#include "voxel.cuh"
#include "twistf.h"

namespace lio {

constexpr int kCubeL = 21, kCubeW = 21, kCubeH = 11, kCubes = kCubeL * kCubeW * kCubeH;

// q * v (Eigen _transformVector) in float, host copy of the device expression
static void rotate_host(const TwistF &t, float vx, float vy, float vz, float &ox, float &oy, float &oz) {
  volatile float ux = t.qy * vz - t.qz * vy, uy = t.qz * vx - t.qx * vz, uz = t.qx * vy - t.qy * vx;
  volatile float ux2 = ux + ux, uy2 = uy + uy, uz2 = uz + uz;
  volatile float cx = t.qy * uz2 - t.qz * uy2, cy = t.qz * ux2 - t.qx * uz2, cz = t.qx * uy2 - t.qy * ux2;
  volatile float ax = ux2 * t.qw, ay = uy2 * t.qw, az = uz2 * t.qw;
  volatile float rx = vx + ax, ry = vy + ay, rz = vz + az;
  ox = rx + cx; oy = ry + cy; oz = rz + cz;
}

// ---- kernels ----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void rotate_dev(float qx, float qy, float qz, float qw, float vx, float vy, float vz, float &ox, float &oy, float &oz) {
  float ux = qy * vz - qz * vy, uy = qz * vx - qx * vz, uz = qx * vy - qy * vx;
  ux += ux; uy += uy; uz += uz;
  const float cx = qy * uz - qz * uy, cy = qz * ux - qx * uz, cz = qx * uy - qy * ux;
  ox = vx + ux * qw + cx; oy = vy + uy * qw + cy; oz = vz + uz * qw + cz;
}

// PointAssociateToMap (po = q * pi + t, :303-314) followed by PointAssociateTobeMapped (po = q^* * (pi - t), :316-323): the
// reference stacks the last features in the map frame and takes them back before the VoxelGrid (:782-800, :1013-1016).
// Both float steps in the reference's order (-fmad=false), the intermediate kept in registers.  The count is read on the
// device and clamped to n_max; CTA 0 publishes the clamped count in n_out for the kernels after it.
__global__ void __launch_bounds__(256)
k_associate(const float4 *__restrict__ in, float4 *__restrict__ out, const int *__restrict__ n_dev, int n_max, int *__restrict__ n_out, TwistF t) {
  int n = *n_dev;
  n = n < 0 ? 0 : (n > n_max ? n_max : n);
  if (blockIdx.x == 0 && threadIdx.x == 0) *n_out = n;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = __ldg(in + i);
  float x, y, z;
  rotate_dev(t.qx, t.qy, t.qz, t.qw, p.x, p.y, p.z, x, y, z);
  x += t.px; y += t.py; z += t.pz;
  float bx, by, bz;
  rotate_dev(-t.qx, -t.qy, -t.qz, t.qw, x - t.px, y - t.py, z - t.pz, bx, by, bz);
  out[i] = make_float4(bx, by, bz, p.w);
}

// int((v + 25.0) / 50.0) + cen, minus one for negatives (:812-819) - double arithmetic like the reference
__device__ __forceinline__ int cube_of(float v, int cen) {
  int c = int(((double)v + 25.0) / 50.0) + cen;
  if ((double)v + 25.0 < 0) --c;
  return c;
}

constexpr int kKeyStride = 8192;   // sort key = cloud * kKeyStride + cube; kCubes (outside the array) sorts last in its cloud
constexpr int kKeyBits = 14;

// UpdateMapDatabase insert, phase 1, over both down-sampled stacks (corner: [0, n0), surf: [n0, n0 + n1)): map-frame point,
// sort key and per-cube add count of every point
__global__ void __launch_bounds__(256)
k_cube_ids(const float4 *__restrict__ ds0, int n0, const float4 *__restrict__ ds1, int n1, TwistF t, int cen_l, int cen_w, int cen_h,
           float4 *__restrict__ mapped, unsigned *__restrict__ key, unsigned *__restrict__ val, int *__restrict__ add, int *__restrict__ n_tot) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *n_tot = n0 + n1;
  if (i >= n0 + n1) return;
  const int w = i >= n0 ? 1 : 0;
  const float4 p = w ? __ldg(ds1 + (i - n0)) : __ldg(ds0 + i);
  float x, y, z;
  rotate_dev(t.qx, t.qy, t.qz, t.qw, p.x, p.y, p.z, x, y, z);
  x += t.px; y += t.py; z += t.pz;
  mapped[i] = make_float4(x, y, z, p.w);
  const int ci = cube_of(x, cen_l), cj = cube_of(y, cen_w), ck = cube_of(z, cen_h);
  const bool inside = ci >= 0 && ci < kCubeL && cj >= 0 && cj < kCubeW && ck >= 0 && ck < kCubeH;
  const int c = inside ? ci + kCubeL * cj + kCubeL * kCubeW * ck : kCubes;
  key[i] = (unsigned)(w * kKeyStride + c);
  val[i] = (unsigned)i;
  if (inside) atomicAdd(add + w * kCubes + c, 1);
}

// phase 2, after the stable sort: the first position of every key's run
__global__ void __launch_bounds__(256) k_run_heads(const unsigned *__restrict__ key, int n, int *__restrict__ start) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const unsigned k = key[s];
  if (s == 0 || key[s - 1] != k) start[k] = s;
}

// phase 3: sorted position s goes to the append position of its cube + its rank in the run - the push_back order of the
// input, because the sort is stable
__global__ void __launch_bounds__(256)
k_scatter_to_cubes(const float4 *__restrict__ mapped, const unsigned *__restrict__ key, const unsigned *__restrict__ val, const int *__restrict__ start,
                   float4 *const *__restrict__ base, int n) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const unsigned k = key[s];
  if ((int)(k % kKeyStride) == kCubes) return;
  base[k][s - start[k]] = __ldg(mapped + val[s]);
}

struct Segment { const float4 *src; int n; int off; };
// concatenation of cube segments (laser_cloud_*_from_map_, :1005-1011); one block range per segment
__global__ void __launch_bounds__(256)
k_gather_segments(const Segment *__restrict__ seg, int nseg, float4 *__restrict__ out) {
  for (int s = blockIdx.y; s < nseg; s += gridDim.y) {
    const Segment sg = seg[s];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < sg.n; i += gridDim.x * blockDim.x) out[sg.off + i] = __ldg(sg.src + i);
  }
}

}  // namespace lio

using namespace lio;

// Pinned staging of one process call (written by the host, read by async copies that complete before the call's last
// synchronisation, or before the first one of the next call).
struct PmStage {
  int cnt_up[2];                        // host-path input counts
  int n_ds[2];                          // read-back: down-sampled stack sizes
  int add[2 * kCubes];                  // read-back: points each cube receives (corner, surf)
  float4 *base[2 * kKeyStride];         // append position of every touched cube, by sort key
  Segment seg[2][256];                  // laser_cloud_{corner,surf}_from_map_ segments
  int vgn[256], vgout[256];             // re-filter input / output counts
};

struct lio_pm {
  struct Cube { float4 *p = nullptr; int n = 0, cap = 0; };
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm = 148;
  int max_points = 0;
  std::vector<Cube> cube[2];           // [0] corner, [1] surf: kCubes descriptors each
  int cen_l = 10, cen_w = 10, cen_h = 5;
  float leaf[2] = {0.2f, 0.4f};
  float min_match_sq_dis = 1.0f, min_plane_dis = 0.2f;
  int max_iter = 10;
  double delta_r_abort = 0.05, delta_t_abort = 0.05;
  TwistF sum, bef, aft, tobe;          // transform_sum_, transform_bef_mapped_, transform_aft_mapped_, transform_tobe_mapped_
  // device scratch
  float4 *d_in[2] = {nullptr, nullptr}, *d_stack[2] = {nullptr, nullptr}, *d_ds[2] = {nullptr, nullptr}, *d_mapped = nullptr, *d_tmp = nullptr;
  float4 *d_map[2] = {nullptr, nullptr};
  int map_cap[2] = {0, 0};
  int *d_cnt = nullptr;                // [0,1] clamped input sizes, [2,3] down-sampled sizes, [4,5] host-path input sizes, [6] insert size, [7] 0
  unsigned *d_key[2] = {nullptr, nullptr}, *d_val[2] = {nullptr, nullptr};   // insert sort ping-pong (2 max_points)
  RadixSortTemp rs;
  int *d_add = nullptr;                // 2 x kCubes
  int *d_start = nullptr;              // 2 x kKeyStride run heads
  float4 **d_base = nullptr;           // 2 x kKeyStride append positions (device mirror of the touched directory entries)
  Segment *d_seg = nullptr;
  int *d_vgout = nullptr;              // per re-filtered cube: output count
  VoxelGrid vg;
  int vg_cap = 0;
  ScanToMapWork stm;
  int stm_cap[3] = {0, 0, 0};
  int last_iters = 0, last_from_map[2] = {0, 0};
  PmStage *h = nullptr;
  CallStats stats;
};

static size_t to_index(int i, int j, int k) { return (size_t)i + (size_t)kCubeL * j + (size_t)kCubeL * kCubeW * k; }
static int cube_of_host(float v, int cen) {
  int c = int(((double)v + 25.0) / 50.0) + cen;
  if ((double)v + 25.0 < 0) --c;
  return c;
}

extern "C" int lio_pm_destroy(lio_pm *m) {
  if (!m) return LIO_OK;
  cudaSetDevice(m->device);
  for (int w = 0; w < 2; ++w) {
    for (lio_pm::Cube &c : m->cube[w]) if (c.p) cudaFree(c.p);
    void *fr[] = {m->d_in[w], m->d_stack[w], m->d_ds[w], m->d_map[w], m->d_key[w], m->d_val[w]};
    for (void *q : fr) if (q) cudaFree(q);
  }
  void *fr[] = {m->d_mapped, m->d_tmp, m->d_cnt, m->d_add, m->d_start, m->d_base, m->d_seg, m->d_vgout};
  for (void *q : fr) if (q) cudaFree(q);
  if (m->h) cudaFreeHost(m->h);
  m->rs.destroy();
  m->vg.destroy();
  m->stm.destroy();
  delete m;
  return LIO_OK;
}

extern "C" int lio_pm_create(int max_points, float corner_filter_size, float surf_filter_size, float min_match_sq_dis, float min_plane_dis,
                             int max_iterations, int device, void *cuda_stream, lio_pm **out) {
  if (!out || max_points < 16 || !(corner_filter_size > 0) || !(surf_filter_size > 0) || max_iterations < 0) return LIO_ERR_INVALID;
  if (lio_device_count() <= 0) return LIO_ERR_NO_DEVICE;
  LIO_CUDA_OK(cudaSetDevice(device));
  lio_pm *m = new (std::nothrow) lio_pm();
  if (!m) return LIO_ERR_INVALID;
  m->device = device; m->stream = (cudaStream_t)cuda_stream; m->max_points = max_points;
  m->leaf[0] = corner_filter_size; m->leaf[1] = surf_filter_size;
  m->min_match_sq_dis = min_match_sq_dis; m->min_plane_dis = min_plane_dis; m->max_iter = max_iterations;
  cudaDeviceGetAttribute(&m->sm, cudaDevAttrMultiProcessorCount, device);
  m->cube[0].assign(kCubes, lio_pm::Cube());
  m->cube[1].assign(kCubes, lio_pm::Cube());
  bool ok = true;
  for (int w = 0; w < 2 && ok; ++w) {
    ok = ok && cudaMalloc(&m->d_in[w], sizeof(float4) * max_points) == cudaSuccess;
    ok = ok && cudaMalloc(&m->d_stack[w], sizeof(float4) * max_points) == cudaSuccess;
    ok = ok && cudaMalloc(&m->d_ds[w], sizeof(float4) * max_points) == cudaSuccess;
    ok = ok && cudaMalloc(&m->d_key[w], sizeof(unsigned) * 2 * max_points) == cudaSuccess;
    ok = ok && cudaMalloc(&m->d_val[w], sizeof(unsigned) * 2 * max_points) == cudaSuccess;
  }
  ok = ok && cudaMalloc(&m->d_mapped, sizeof(float4) * 2 * max_points) == cudaSuccess;
  ok = ok && cudaMalloc(&m->d_cnt, sizeof(int) * 8) == cudaSuccess && cudaMemset(m->d_cnt, 0, sizeof(int) * 8) == cudaSuccess;
  ok = ok && m->rs.init(2 * max_points) == 0;
  ok = ok && cudaMalloc(&m->d_add, sizeof(int) * 2 * kCubes) == cudaSuccess;
  ok = ok && cudaMalloc(&m->d_start, sizeof(int) * 2 * kKeyStride) == cudaSuccess;
  ok = ok && cudaMalloc(&m->d_base, sizeof(float4 *) * 2 * kKeyStride) == cudaSuccess;
  ok = ok && cudaMalloc(&m->d_seg, sizeof(Segment) * 256) == cudaSuccess;
  ok = ok && cudaMalloc(&m->d_vgout, sizeof(int) * 256) == cudaSuccess;
  ok = ok && cudaMallocHost(&m->h, sizeof(PmStage)) == cudaSuccess;
  m->vg_cap = max_points;
  ok = ok && cudaMalloc(&m->d_tmp, sizeof(float4) * m->vg_cap) == cudaSuccess;
  ok = ok && m->vg.init(m->vg_cap) == 0;
  if (!ok) { lio_set_last_error(__FILE__, __LINE__, "lio_pm_create: device allocation failed"); lio_pm_destroy(m); return LIO_ERR_CUDA; }
  *out = m;
  return LIO_OK;
}

// ---- host-side directory logic (the reference's own index arithmetic) ---------------------------------------------------
static void pm_recentre(lio_pm *m, float px, float py, float pz, int &ci, int &cj, int &ck) {   // :812-931
  ci = cube_of_host(px, m->cen_l); cj = cube_of_host(py, m->cen_w); ck = cube_of_host(pz, m->cen_h);
  auto shift = [&](int axis, int dir) {  // dir +1: contents move towards higher indices, the low face is cleared
    const int n[3] = {kCubeL, kCubeW, kCubeH};
    int idx[3];
    for (idx[(axis + 1) % 3] = 0; idx[(axis + 1) % 3] < n[(axis + 1) % 3]; ++idx[(axis + 1) % 3])
      for (idx[(axis + 2) % 3] = 0; idx[(axis + 2) % 3] < n[(axis + 2) % 3]; ++idx[(axis + 2) % 3]) {
        if (dir > 0) {
          for (int a = n[axis] - 1; a >= 1; --a) {
            idx[axis] = a; const size_t ia = to_index(idx[0], idx[1], idx[2]);
            idx[axis] = a - 1; const size_t ib = to_index(idx[0], idx[1], idx[2]);
            std::swap(m->cube[0][ia], m->cube[0][ib]); std::swap(m->cube[1][ia], m->cube[1][ib]);
          }
          idx[axis] = 0;
        } else {
          for (int a = 0; a < n[axis] - 1; ++a) {
            idx[axis] = a; const size_t ia = to_index(idx[0], idx[1], idx[2]);
            idx[axis] = a + 1; const size_t ib = to_index(idx[0], idx[1], idx[2]);
            std::swap(m->cube[0][ia], m->cube[0][ib]); std::swap(m->cube[1][ia], m->cube[1][ib]);
          }
          idx[axis] = n[axis] - 1;
        }
        const size_t ic = to_index(idx[0], idx[1], idx[2]);
        m->cube[0][ic].n = 0; m->cube[1][ic].n = 0;   // clear(): the HBM segment is kept for re-use
      }
  };
  while (ci < 3) { shift(0, +1); ++ci; ++m->cen_l; }
  while (ci >= kCubeL - 3) { shift(0, -1); --ci; --m->cen_l; }
  while (cj < 3) { shift(1, +1); ++cj; ++m->cen_w; }
  while (cj >= kCubeW - 3) { shift(1, -1); --cj; --m->cen_w; }
  while (ck < 3) { shift(2, +1); ++ck; ++m->cen_h; }
  while (ck >= kCubeH - 3) { shift(2, -1); --ck; --m->cen_h; }
}

static void pm_select(const lio_pm *m, float px, float py, float pz, const float z[3], int ci, int cj, int ck, std::vector<size_t> &valid) {   // :944-1003
  valid.clear();
  for (int i = ci - 2; i <= ci + 2; ++i)
    for (int j = cj - 2; j <= cj + 2; ++j)
      for (int k = ck - 2; k <= ck + 2; ++k) {
        if (!(i >= 0 && i < kCubeL && j >= 0 && j < kCubeW && k >= 0 && k < kCubeH)) continue;
        const float center_x = 50.0f * (i - m->cen_l), center_y = 50.0f * (j - m->cen_w), center_z = 50.0f * (k - m->cen_h);
        bool is_in_laser_fov = false;
        for (int ii = -1; ii <= 1; ii += 2)
          for (int jj = -1; jj <= 1; jj += 2)
            for (int kk = -1; kk <= 1; kk += 2) {
              const float cx = center_x + 25.0f * ii, cy = center_y + 25.0f * jj, cz = center_z + 25.0f * kk;
              const float d0 = px - cx, d1 = py - cy, d2 = pz - cz;
              volatile float s1 = d0 * d0; s1 = s1 + d1 * d1; s1 = s1 + d2 * d2;
              const float e0 = z[0] - cx, e1 = z[1] - cy, e2 = z[2] - cz;
              volatile float s2 = e0 * e0; s2 = s2 + e1 * e1; s2 = s2 + e2 * e2;
              const float squared_side1 = s1, squared_side2 = s2;
              const float check1 = 100.0f + squared_side1 - squared_side2 - 10.0f * std::sqrt(3.0f) * std::sqrt(squared_side1);
              const float check2 = 100.0f + squared_side1 - squared_side2 + 10.0f * std::sqrt(3.0f) * std::sqrt(squared_side1);
              if (check1 < 0 && check2 > 0) is_in_laser_fov = true;
            }
        if (is_in_laser_fov) valid.push_back(to_index(i, j, k));
      }
}

// Segments (and the pulled maps) come from the stream-ordered allocator: allocation, copy of the old contents and release of
// the old segment are all enqueued on the context's stream, so growing a cube costs the host no synchronisation.
static int pm_grow(lio_pm *m, lio_pm::Cube &c, int need) {
  if (need <= c.cap) return LIO_OK;
  int cap = std::max(1024, c.cap);
  while (cap < need) cap *= 2;
  float4 *p = nullptr;
  LIO_CUDA_OK(cudaMallocAsync((void **)&p, sizeof(float4) * cap, m->stream));
  if (c.p && c.n > 0) LIO_CUDA_OK(cudaMemcpyAsync(p, c.p, sizeof(float4) * c.n, cudaMemcpyDeviceToDevice, m->stream));
  if (c.p) LIO_CUDA_OK(cudaFreeAsync(c.p, m->stream));
  c.p = p; c.cap = cap;
  return LIO_OK;
}

// laser_cloud_*_from_map_: concatenate the valid cubes (in `valid` order) into d_map[w]
static int pm_from_map(lio_pm *m, const std::vector<size_t> &valid, int w, int &total) {
  Segment *seg = m->h->seg[w];
  int nseg = 0;
  total = 0;
  for (size_t v : valid) {
    const lio_pm::Cube &c = m->cube[w][v];
    if (c.n > 0) {
      if (nseg == 256) return LIO_ERR_CAPACITY;
      seg[nseg++] = Segment{c.p, c.n, total};
      total += c.n;
    }
  }
  if (total > m->map_cap[w]) {
    if (m->d_map[w]) LIO_CUDA_OK(cudaFreeAsync(m->d_map[w], m->stream));
    m->d_map[w] = nullptr;
    m->map_cap[w] = std::max(2 * total, 1 << 16);
    LIO_CUDA_OK(cudaMallocAsync((void **)&m->d_map[w], sizeof(float4) * m->map_cap[w], m->stream));
  }
  if (nseg == 0) return LIO_OK;
  LIO_CUDA_OK(stats_h2d(m->stats, m->d_seg, seg, sizeof(Segment) * nseg, m->stream));
  k_gather_segments<<<dim3(16, (unsigned)nseg), 256, 0, m->stream>>>(m->d_seg, nseg, m->d_map[w]);
  ++m->stats.launches;
  return LIO_OK;
}

// UpdateMapDatabase (:1112-1208) with margin centre == current centre (the valid list was computed in this call)
static int pm_update(lio_pm *m, const std::vector<size_t> &valid, const int n_ds[2]) {
  cudaStream_t st = m->stream;
  CallStats &S = m->stats;
  PmStage *h = m->h;
  // the cubes re-filtered after the insert (corner then surf of every valid cube), each with its own bounding box like
  // pcl::VoxelGrid on that cube's cloud
  std::vector<size_t> refilter;
  for (size_t index : valid) {
    int li, lj, lk;
    { int residual = (int)(index % (kCubeL * kCubeW)); lk = (int)(index / (kCubeL * kCubeW)); lj = residual / kCubeL; li = residual % kCubeL; }
    const float center_x = 50.0f * (li - m->cen_l), center_y = 50.0f * (lj - m->cen_w), center_z = 50.0f * (lk - m->cen_h);
    const int ci = cube_of_host(center_x, m->cen_l), cj = cube_of_host(center_y, m->cen_w), ck = cube_of_host(center_z, m->cen_h);
    if (!(ci >= 0 && ci < kCubeL && cj >= 0 && cj < kCubeW && ck >= 0 && ck < kCubeH)) continue;
    refilter.push_back(to_index(ci, cj, ck));
  }
  const int n = n_ds[0] + n_ds[1];
  if (n > 0) {
    // insert: cube ids + add counts, stable sort of (cloud, cube | input index), run heads; the add counts come back
    LIO_CUDA_OK(cudaMemsetAsync(m->d_add, 0, sizeof(int) * 2 * kCubes, st));
    const int nb = (n + 255) / 256;
    k_cube_ids<<<nb, 256, 0, st>>>(m->d_ds[0], n_ds[0], m->d_ds[1], n_ds[1], m->tobe, m->cen_l, m->cen_w, m->cen_h, m->d_mapped, m->d_key[0],
                                   m->d_val[0], m->d_add, m->d_cnt + 6);
    int launches = 1;
    const int which = radix_sort_pairs(m->d_key[0], m->d_val[0], m->d_key[1], m->d_val[1], m->d_cnt + 6, n, kKeyBits, m->rs, st, &launches);
    if (which < 0) { lio_set_last_error(__FILE__, __LINE__, "cube insert: sort workspace too small"); return LIO_ERR_CAPACITY; }
    const unsigned *skey = m->d_key[which], *sval = m->d_val[which];
    k_run_heads<<<nb, 256, 0, st>>>(skey, n, m->d_start);
    ++launches;
    S.launches += launches;
    LIO_CUDA_OK(stats_d2h(S, h->add, m->d_add, sizeof(int) * 2 * kCubes, st));
    LIO_CUDA_OK(stats_sync(S, st));
    // grow the receiving segments, then the re-filter workspace to the largest cube it will see - before anything moves, so
    // a failure leaves the map as it was
    int need_vg = 0;
    for (int w = 0; w < 2; ++w)
      for (int c = 0; c < kCubes; ++c)
        if (h->add[w * kCubes + c]) { int rc = pm_grow(m, m->cube[w][c], m->cube[w][c].n + h->add[w * kCubes + c]); if (rc != LIO_OK) return rc; }
    for (size_t idx : refilter)
      for (int w = 0; w < 2; ++w) need_vg = std::max(need_vg, m->cube[w][idx].n + h->add[w * kCubes + idx]);
    if (need_vg > m->vg_cap) {
      int cap = m->vg_cap;
      while (cap < need_vg) cap *= 2;
      ++S.syncs;   // cudaFree synchronises the device
      m->vg.destroy();
      if (m->d_tmp) cudaFree(m->d_tmp);
      m->d_tmp = nullptr;
      m->vg_cap = 0;
      if (cudaMalloc(&m->d_tmp, sizeof(float4) * cap) != cudaSuccess || m->vg.init(cap) != 0) {
        lio_set_last_error(__FILE__, __LINE__, "cube re-filter workspace allocation failed");
        return LIO_ERR_CUDA;
      }
      m->vg_cap = cap;
    }
    // append positions of the touched cubes, one contiguous key range per cloud
    for (int w = 0; w < 2; ++w) {
      int lo = kCubes, hi = -1;
      for (int c = 0; c < kCubes; ++c)
        if (h->add[w * kCubes + c]) {
          lo = std::min(lo, c); hi = c;
          h->base[w * kKeyStride + c] = m->cube[w][c].p + m->cube[w][c].n;
        }
      if (hi >= lo) LIO_CUDA_OK(stats_h2d(S, m->d_base + w * kKeyStride + lo, h->base + w * kKeyStride + lo, sizeof(float4 *) * (hi - lo + 1), st));
    }
    k_scatter_to_cubes<<<nb, 256, 0, st>>>(m->d_mapped, skey, sval, m->d_start, m->d_base, n);
    ++S.launches;
    for (int w = 0; w < 2; ++w)
      for (int c = 0; c < kCubes; ++c) m->cube[w][c].n += h->add[w * kCubes + c];
  }
  struct Job { int w; size_t idx; };
  std::vector<Job> jobs;
  for (size_t idx : refilter)
    for (int w = 0; w < 2; ++w) if (m->cube[w][idx].n > 0) jobs.push_back(Job{w, idx});
  for (size_t b0 = 0; b0 < jobs.size(); b0 += 256) {
    const size_t b1 = std::min(jobs.size(), b0 + 256);
    // input count through d_vgout[j] itself (read before the filter overwrites it with the output count)
    for (size_t j = b0; j < b1; ++j) h->vgn[j - b0] = m->cube[jobs[j].w][jobs[j].idx].n;
    LIO_CUDA_OK(stats_h2d(S, m->d_vgout, h->vgn, sizeof(int) * (b1 - b0), st));
    int launches = 0;
    for (size_t j = b0; j < b1; ++j) {
      lio_pm::Cube &c = m->cube[jobs[j].w][jobs[j].idx];
      int rc = m->vg.run(c.p, m->d_vgout + (j - b0), c.n, m->leaf[jobs[j].w], m->d_tmp, m->vg_cap, m->d_vgout + (j - b0), nullptr, st, &launches);
      if (rc != LIO_OK) return rc;
      LIO_CUDA_OK(cudaMemcpyAsync(c.p, m->d_tmp, sizeof(float4) * c.n, cudaMemcpyDeviceToDevice, st));   // output <= input count
    }
    S.launches += launches;
    LIO_CUDA_OK(stats_d2h(S, h->vgout, m->d_vgout, sizeof(int) * (b1 - b0), st));
    LIO_CUDA_OK(stats_sync(S, st));
    for (size_t j = b0; j < b1; ++j) m->cube[jobs[j].w][jobs[j].idx].n = h->vgout[j - b0];
  }
  return LIO_OK;
}

// PointMapping::Process (:765-1052), imu_inited_ == false, num_stack_frames_ == 1, on device clouds: src[w] with a device
// count clamped to n_max[w] on the device.  Shared by the host and device entries.
static int pm_core(lio_pm *m, const float4 *const src[2], const int *const n_dev[2], const int n_max[2], const float transform_sum7[7],
                   float transform_tobe_mapped7[7], int info3[3]) {
  cudaStream_t st = m->stream;
  CallStats &S = m->stats;
  m->sum = TwistF{transform_sum7[0], transform_sum7[1], transform_sum7[2], transform_sum7[3], transform_sum7[4], transform_sum7[5], transform_sum7[6]};
  m->tobe = twist_mul(m->tobe, twist_mul(twist_inverse(m->bef), m->sum));   // TransformAssociateToMap :753-756
  for (int w = 0; w < 2; ++w) {
    if (n_max[w] == 0) continue;
    k_associate<<<(n_max[w] + 255) / 256, 256, 0, st>>>(src[w], m->d_stack[w], n_dev[w], n_max[w], m->d_cnt + w, m->tobe);
    ++S.launches;
  }
  float z[3];
  {  // point_on_z_axis_ = tobe * (0, 0, 10)
    rotate_host(m->tobe, 0.0f, 0.0f, 10.0f, z[0], z[1], z[2]);
    z[0] += m->tobe.px; z[1] += m->tobe.py; z[2] += m->tobe.pz;
  }
  int ci, cj, ck;
  pm_recentre(m, m->tobe.px, m->tobe.py, m->tobe.pz, ci, cj, ck);
  std::vector<size_t> valid;
  pm_select(m, m->tobe.px, m->tobe.py, m->tobe.pz, z, ci, cj, ck, valid);
  int K[2] = {0, 0};
  for (int w = 0; w < 2; ++w) { int rc = pm_from_map(m, valid, w, K[w]); if (rc != LIO_OK) return rc; }
  m->last_from_map[0] = K[0]; m->last_from_map[1] = K[1];
  // down-sample the stacks
  int launches = 0;
  for (int w = 0; w < 2; ++w) {
    if (n_max[w] == 0) { LIO_CUDA_OK(cudaMemsetAsync(m->d_cnt + 2 + w, 0, sizeof(int), st)); continue; }
    int rc = m->vg.run(m->d_stack[w], m->d_cnt + w, n_max[w], m->leaf[w], m->d_ds[w], m->max_points, m->d_cnt + 2 + w, nullptr, st, &launches);
    if (rc != LIO_OK) return rc;
  }
  S.launches += launches;
  LIO_CUDA_OK(stats_d2h(S, m->h->n_ds, m->d_cnt + 2, sizeof(int) * 2, st));
  LIO_CUDA_OK(stats_sync(S, st));
  const int n_ds[2] = {m->h->n_ds[0], m->h->n_ds[1]};
  // OptimizeTransformTobeMapped against the pulled map
  const bool optimised = !(K[0] <= 10 || K[1] <= 100);
  m->last_iters = 0;
  if (optimised && m->max_iter > 0) {
    if (K[0] > m->stm_cap[0] || K[1] > m->stm_cap[1] || n_ds[0] + n_ds[1] > m->stm_cap[2]) {
      if (m->stm_cap[0] > 0) ++S.syncs;   // cudaFree of the old workspace synchronises the device
      m->stm.destroy();
      m->stm_cap[0] = std::max(2 * K[0], 1 << 15); m->stm_cap[1] = std::max(2 * K[1], 1 << 16); m->stm_cap[2] = std::max(2 * (n_ds[0] + n_ds[1]), 1 << 15);
      if (m->stm.init(m->stm_cap[0], m->stm_cap[1], m->stm_cap[2]) != 0) { lio_set_last_error(__FILE__, __LINE__, "scan-to-map workspace allocation failed"); return LIO_ERR_CUDA; }
    }
    float tf7[7] = {m->tobe.qx, m->tobe.qy, m->tobe.qz, m->tobe.qw, m->tobe.px, m->tobe.py, m->tobe.pz};
    int rc = scan_to_map_run(m->stm, m->d_map[0], K[0], m->d_map[1], K[1], m->d_ds[0], m->d_cnt + 2, std::max(n_ds[0], 1), m->d_ds[1], m->d_cnt + 3,
                             std::max(n_ds[1], 1), tf7, m->min_match_sq_dis, m->min_plane_dis, m->max_iter, m->delta_r_abort, m->delta_t_abort, 0, nullptr,
                             &m->last_iters, m->sm, st, &S);
    if (rc != LIO_OK) return rc;
    m->tobe = TwistF{tf7[0], tf7[1], tf7[2], tf7[3], tf7[4], tf7[5], tf7[6]};
  }
  if (optimised) { m->bef = m->sum; m->aft = m->tobe; }   // TransformUpdate sits behind the optimiser's early return (:327-329, :716)
  int rc = pm_update(m, valid, n_ds);
  if (rc != LIO_OK) return rc;
  LIO_CUDA_OK(cudaGetLastError());
  if (transform_tobe_mapped7) {
    transform_tobe_mapped7[0] = m->tobe.qx; transform_tobe_mapped7[1] = m->tobe.qy; transform_tobe_mapped7[2] = m->tobe.qz; transform_tobe_mapped7[3] = m->tobe.qw;
    transform_tobe_mapped7[4] = m->tobe.px; transform_tobe_mapped7[5] = m->tobe.py; transform_tobe_mapped7[6] = m->tobe.pz;
  }
  if (info3) { info3[0] = m->last_iters; info3[1] = K[0]; info3[2] = K[1]; }
  return LIO_OK;
}

// Host arrays of n x 4 floats: uploaded into the context's buffers, then the same core.
extern "C" int lio_pm_process_host(lio_pm *m, const float *corner_last, int nc, const float *surf_last, int ns, const float transform_sum7[7],
                                   float transform_tobe_mapped7[7], int info3[3]) {
  if (!m || !transform_sum7 || nc < 0 || ns < 0 || (nc > 0 && !corner_last) || (ns > 0 && !surf_last)) return LIO_ERR_INVALID;
  if (nc > m->max_points || ns > m->max_points) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(m->device));
  cudaStream_t st = m->stream;
  m->stats.reset();
  const float *src[2] = {corner_last, surf_last};
  const int nin[2] = {nc, ns};
  for (int w = 0; w < 2; ++w) {
    m->h->cnt_up[w] = nin[w];
    if (nin[w]) LIO_CUDA_OK(stats_h2d(m->stats, m->d_in[w], src[w], sizeof(float4) * nin[w], st));
  }
  LIO_CUDA_OK(stats_h2d(m->stats, m->d_cnt + 4, m->h->cnt_up, sizeof(int) * 2, st));
  const float4 *const din[2] = {m->d_in[0], m->d_in[1]};
  const int *const dn[2] = {m->d_cnt + 4, m->d_cnt + 5};
  return pm_core(m, din, dn, nin, transform_sum7, transform_tobe_mapped7, info3);
}

extern "C" int lio_pm_process_dev(lio_pm *m, const lio_dev_cloud *corner_last, const lio_dev_cloud *surf_last, const float transform_sum7[7],
                                  float transform_tobe_mapped7[7], int info3[3]) {
  if (!m || !transform_sum7 || !corner_last || !surf_last) return LIO_ERR_INVALID;
  const lio_dev_cloud *c[2] = {corner_last, surf_last};
  for (int w = 0; w < 2; ++w)
    if (c[w]->n_max < 0 || (c[w]->n_max > 0 && (!c[w]->xyzi || !c[w]->n_dev))) return LIO_ERR_INVALID;
  if (corner_last->n_max > m->max_points || surf_last->n_max > m->max_points) {
    lio_set_last_error(__FILE__, __LINE__, "lio_pm_process_dev: n_max exceeds the max_points given to lio_pm_create");
    return LIO_ERR_CAPACITY;
  }
  LIO_CUDA_OK(cudaSetDevice(m->device));
  m->stats.reset();
  const float4 *const src[2] = {reinterpret_cast<const float4 *>(c[0]->xyzi), reinterpret_cast<const float4 *>(c[1]->xyzi)};
  const int *const dn[2] = {c[0]->n_max > 0 ? c[0]->n_dev : m->d_cnt + 7, c[1]->n_max > 0 ? c[1]->n_dev : m->d_cnt + 7};
  const int nmax[2] = {c[0]->n_max, c[1]->n_max};
  return pm_core(m, src, dn, nmax, transform_sum7, transform_tobe_mapped7, info3);
}

extern "C" int lio_pm_last_stats(lio_pm *m, long long out[4]) {
  if (!m || !out) return LIO_ERR_INVALID;
  out[0] = m->stats.launches; out[1] = m->stats.syncs; out[2] = m->stats.h2d; out[3] = m->stats.d2h;
  return LIO_OK;
}

extern "C" int lio_pm_map_centre(lio_pm *m, int centre3[3]) {
  if (!m || !centre3) return LIO_ERR_INVALID;
  centre3[0] = m->cen_l; centre3[1] = m->cen_w; centre3[2] = m->cen_h;
  return LIO_OK;
}

extern "C" int lio_pm_cube_size(lio_pm *m, int cube_index, int which, int *n) {
  if (!m || !n || cube_index < 0 || cube_index >= kCubes || which < 0 || which > 1) return LIO_ERR_INVALID;
  *n = m->cube[which][cube_index].n;
  return LIO_OK;
}

extern "C" int lio_pm_cube_download(lio_pm *m, int cube_index, int which, float *out_xyzi, int cap) {
  if (!m || !out_xyzi || cube_index < 0 || cube_index >= kCubes || which < 0 || which > 1) return LIO_ERR_INVALID;
  const lio_pm::Cube &c = m->cube[which][cube_index];
  if (c.n > cap) return LIO_ERR_CAPACITY;
  LIO_CUDA_OK(cudaSetDevice(m->device));
  if (c.n > 0) LIO_CUDA_OK(cudaMemcpyAsync(out_xyzi, c.p, sizeof(float4) * c.n, cudaMemcpyDeviceToHost, m->stream));
  LIO_CUDA_OK(cudaStreamSynchronize(m->stream));
  return LIO_OK;
}
