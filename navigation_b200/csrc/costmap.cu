// costmap.cu -- Path A host side: the device-resident layered costmap behind the navgpu_costmap_* C ABI.
//
// Mirrors costmap_2d::LayeredCostmap + its Layer plugins (reference file:line cited per function).  Everything that
// touches grid cells runs in the kernels of costmap_kernels.cuh; the host keeps only the scalar state the reference
// keeps in its objects (origins, parameters, cached tables, flags) and sequences the kernels of one update cycle.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <vector>

#include "costmap_kernels.cuh"
#include "fleet_costmap.cuh"
#include "fleet_costmap_kernels.cuh"
#include "inflate_propagate.cuh"
#include "mirror_kernels.cuh"

namespace navgpu {

struct Pt {
  double x, y;
};

// calculateMinAndMaxDistances, src/footprint.cpp:41-67 (pure scalar geometry, evaluated once per footprint change)
static double dist2d(double x0, double y0, double x1, double y1) { return hypot(x1 - x0, y1 - y0); }
static double distance_to_line(double pX, double pY, double x0, double y0, double x1, double y1) {  // costmap_math.cpp:32-63
  double A = pX - x0, B = pY - y0, C = x1 - x0, D = y1 - y0;
  double dot = A * C + B * D, len_sq = C * C + D * D, param = dot / len_sq;
  double xx, yy;
  if (param < 0) { xx = x0; yy = y0; }
  else if (param > 1) { xx = x1; yy = y1; }
  else { xx = x0 + param * C; yy = y0 + param * D; }
  return dist2d(pX, pY, xx, yy);
}
void footprint_radii(const std::vector<Pt>& fp, double& mn, double& mx) {
  mn = std::numeric_limits<double>::max();
  mx = 0.0;
  if (fp.size() <= 2) return;
  for (size_t i = 0; i < fp.size(); ++i) {
    const Pt& a = fp[i];
    const Pt& b = fp[(i + 1) % fp.size()];
    double vd = dist2d(0, 0, a.x, a.y), ed = distance_to_line(0, 0, a.x, a.y, b.x, b.y);
    mn = std::min(mn, std::min(vd, ed));
    mx = std::max(mx, std::max(vd, ed));
  }
}

// InflationLayer::computeCost / computeCaches (inflation_layer.h:114-129, plugins/inflation_layer.cpp:295-328):
// evaluated on the host with the reference formula (hypot, exp of the host libm) so the tables are bit-identical.
struct CostTables {
  unsigned R = 0;
  std::vector<uint8_t> costs;  // (R+2)^2, [dx][dy]
  std::vector<double> dists;
  std::vector<uint8_t> by_d2;  // R*R+1: cost by squared distance
  std::vector<uint16_t> rank;  // (R+2)^2: dense rank of dists (1 = distance 0), 0xffff where dists > R (mode 1)
  int reach2 = 0;              // largest squared distance with a non-zero cost
  bool ambiguous = false;      // two (dx,dy) with equal dx^2+dy^2 but different cached cost (never seen in practice)
};
static uint8_t compute_cost(double distance, double resolution, double inscribed, double weight) {
  unsigned char cost = 0;
  if (distance == 0) cost = kLethal;
  else if (distance * resolution <= inscribed) cost = kInscribed;
  else {
    double euclidean_distance = distance * resolution;
    double factor = exp(-1.0 * weight * (euclidean_distance - inscribed));
    cost = (unsigned char)((kInscribed - 1) * factor);
  }
  return cost;
}
static int reach_of(const std::vector<uint8_t>& by_d2) {
  int reach2 = 0;
  for (size_t d2 = 0; d2 < by_d2.size(); ++d2)
    if (by_d2[d2] != 0) reach2 = (int)d2;
  return reach2;
}
void build_tables(CostTables& t, unsigned R, double resolution, double inscribed, double weight) {
  t.R = R;
  const unsigned n = R + 2;
  t.costs.assign(size_t(n) * n, 0);
  t.dists.assign(size_t(n) * n, 0.0);
  t.by_d2.assign(size_t(R) * R + 1, 0);
  std::vector<int> seen(size_t(R) * R + 1, 0);
  t.ambiguous = false;
  for (unsigned i = 0; i < n; ++i)
    for (unsigned j = 0; j < n; ++j) {
      double d = hypot(i, j);
      t.dists[i * n + j] = d;
      uint8_t c = compute_cost(d, resolution, inscribed, weight);
      t.costs[i * n + j] = c;
      unsigned d2 = i * i + j * j;
      // the reference enqueues a cell only while cached_distances_ <= cell_inflation_radius_ (:284-287)
      if (d2 <= R * R) {
        if (d > (double)R) t.ambiguous = true;
        if (seen[d2] && t.by_d2[d2] != c) t.ambiguous = true;
        seen[d2] = 1;
        t.by_d2[d2] = c;
      } else if (!(d > (double)R)) {
        t.ambiguous = true;
      }
    }
  t.reach2 = reach_of(t.by_d2);
  // mode 1 orders pops by the cached double itself (inflation_layer.h:77-80): equal doubles <=> equal ranks
  std::vector<double> vals;
  for (double d : t.dists)
    if (!(d > (double)R)) vals.push_back(d);
  std::sort(vals.begin(), vals.end());
  vals.erase(std::unique(vals.begin(), vals.end()), vals.end());
  t.rank.assign(size_t(n) * n, 0xffff);
  for (size_t i = 0; i < t.dists.size(); ++i)
    if (!(t.dists[i] > (double)R))
      t.rank[i] = (uint16_t)(1 + (std::lower_bound(vals.begin(), vals.end(), t.dists[i]) - vals.begin()));
}

static unsigned cell_distance(double world_dist, double resolution) {  // Costmap2D::cellDistance, costmap_2d.cpp:181-185
  double cells_dist = std::max(0.0, ceil(world_dist / resolution));
  return (unsigned int)cells_dist;
}

struct HostObs {
  double ox, oy, oz, obstacle_range, raytrace_range;
  int first_point, n_points;
  bool marking, clearing;
};

struct Layer {
  int kind = 0;  // 0 grid, 1 obstacle, 2 inflation
  bool enabled = true;
  // cost layers (CostmapLayer): own grid with own origin
  uint8_t* grid[2] = {nullptr, nullptr};
  int cur = 0;
  double ox = 0, oy = 0;
  uint8_t def = 0;
  // grid layer
  int policy = 0;
  unsigned ux = 0, uy = 0, uw = 0, uh = 0;
  bool updated = false;
  // obstacle layer
  int combination_method = 1;
  bool footprint_clearing = true;
  double max_obstacle_height = 2.0;
  std::vector<HostObs> obs;
  std::vector<DevObs> h_clear, h_mark;  // host copies of the device tables (they also travel as kernel parameters)
  DevObs* d_clear = nullptr;
  DevObs* d_mark = nullptr;
  float* d_xyz = nullptr;
  long long* d_mark_cells = nullptr;  // scratch of k_obstacle_update: one prepared cell offset per marking point
  size_t xyz_capacity = 0, obs_capacity = 0, mark_cells_capacity = 0;
  char* d_scan = nullptr;  // staging of navgpu_obstacle_set_scans: ScanRec records + ranges
  char* h_stage = nullptr;  // pinned staging of navgpu_obstacle_set_observations' uploads
  size_t stage_capacity = 0;
  cudaEvent_t ev_stage = nullptr;
  size_t scan_capacity = 0;
  int n_clear = 0, n_mark = 0, total_rays = 0, total_marks = 0;
  uint8_t* d_tile_used = nullptr;  // MergeLayers::used (plain obstacle layers of non-rolling, FREE_SPACE-default costmaps)
  // world box of every sensor origin and observation point (rays and marks stay inside it); valid only when the
  // points were seen on the host (navgpu_obstacle_set_observations)
  bool touch_box_valid = false;
  double tbx0 = 0, tby0 = 0, tbx1 = 0, tby1 = 0;
  std::vector<Pt> transformed_footprint;
  // voxel layer (an obstacle layer with columns of 16 voxels, plugins/voxel_layer.cpp)
  bool voxel = false;
  VoxelGeom vg{0.0, 0.2, 10u, 21u, 0u};
  uint32_t* vox[2] = {nullptr, nullptr};
  // inflation layer
  double radius = 0, weight = 0, inscribed = 0;
  bool need_reinflation = false;
  int mode = 0;
  CostTables tables;
  uint8_t* d_cost_d2 = nullptr;
  size_t cost_d2_capacity = 0;
  uint16_t* d_rank = nullptr;   // mode 1: CostTables::rank and ::costs on the device
  uint8_t* d_cost2d = nullptr;
  size_t table2d_capacity = 0;
  bool tables_dirty = true;
};

}  // namespace navgpu

using namespace navgpu;

struct navgpu_costmap {
  int device = 0;
  cudaStream_t stream = nullptr;
  unsigned sx = 0, sy = 0, pitch = 0;
  double res = 0, ox = 0, oy = 0;
  bool rolling = false, track_unknown = false;
  uint8_t def = 0;
  uint8_t* master[2] = {nullptr, nullptr};
  int cur = 0;
  std::vector<Layer> layers;
  std::vector<Pt> footprint;
  double inscribed = 0, circumscribed = 0;
  DevBox* d_boxes = nullptr;
  InflationBoundsState* d_infl = nullptr;
  DevWindow* d_win = nullptr;
  DevWindow* h_win = nullptr;  // pinned
  unsigned* d_ticket = nullptr;  // k_obstacle_update's "last CTA" counter
  unsigned* d_obst_done = nullptr;  // ObstacleArgs::done_flag
  unsigned obst_epoch = 0;
  int8_t* d_occupancy = nullptr;  // packed window for navgpu_costmap_get_window_occupancy
  size_t occupancy_capacity = 0;
  uint16_t* d_seeds = nullptr;  // seed bitmask of the fast sweep (k_merge_seed -> k_inflate)
  size_t seeds_capacity = 0;
  unsigned* d_tile_ready = nullptr;  // early mode: per k_merge_seed tile, the sweep number that last completed it
  unsigned sweep_epoch = 0;
  int sm_count = 0;
  // inflation mode 1 (k_inflate_propagate): per-cell state + two frontier lists, barrier / round control
  uint32_t* d_prop_state = nullptr;
  PropCtl* d_prop_ctl = nullptr;
  int prop_max_blocks = 0;
  size_t prop_smem_set = 0;
  int win[4] = {0, 0, 0, 0};
  bool poly_attr_set = false;
  bool profile = false;
  bool force_generic = false;  // tests: exercise the generic sweep kernel also for R <= 32
  cudaEvent_t ev_sweep[2] = {nullptr, nullptr};
  cudaEvent_t ev_mid = nullptr;  // between k_merge_seed and k_inflate
  cudaEvent_t ev_cycle[2] = {nullptr, nullptr};
  // host mirror kept in sync by navgpu_costmap_get_changed (mirror_kernels.cuh)
  uint8_t* d_shadow = nullptr;           // what the host mirror holds
  const uint8_t* mirror_host = nullptr;  // the host grid the shadow describes
  uint32_t mirror_host_pitch = 0;
  bool shadow_valid = false;
  uint8_t* h_mirror_stage = nullptr;     // mapped pinned: changed tiles, compacted
  unsigned* h_mirror_tiles = nullptr;    // mapped pinned: their tile numbers
  MirrorCtl* h_mirror_ctl = nullptr;     // mapped pinned
  unsigned mirror_seq = 0;               // MirrorCtl::seq of the last k_mirror_diff
  // InflateArgs::done of the sweep that was enqueued last, if it publishes per-tile completion (0: it does not)
  unsigned* d_inflate_done = nullptr;
  size_t inflate_done_capacity = 0;
  unsigned inflate_done_epoch = 0;
  int inflate_done_pitch = 0;
  unsigned* d_mirror_counters = nullptr;
  unsigned mirror_capacity = 0;
  // where the master grid can differ from the shadow (MirrorArgs::dirty / all / hx0..):
  DevWindow* d_mirror_dirty = nullptr;  // accumulated by finalize_bounds, emptied by k_mirror_diff
  bool mirror_all = true;               // something other than an update cycle wrote the master grid (upload, roll)
  bool content_changed = true;          // layer contents / parameters changed by a call since the last update cycle
  bool master_clean = false;            // the last cycle recomputed the whole map: the grid is a pure function of the layers
  bool refine_valid = false;            // every cycle since the last get_changed changed cells only inside refine box
  int refine[4] = {0, 0, 0, 0};         // x0, xn, y0, yn (empty: xn <= x0)

  size_t bytes() const { return size_t(pitch) * sy; }
  Geom geom(double gox, double goy) const { return Geom{sx, sy, pitch, res, gox, goy}; }
  double size_m_x() const { return (sx - 1 + 0.5) * res; }  // Costmap2D::getSizeInMetersX, costmap_2d.cpp:440-443
  double size_m_y() const { return (sy - 1 + 0.5) * res; }
};

namespace {

int use_device(navgpu_costmap* h) {
  NAVGPU_CUDA(cudaSetDevice(h->device));
  return NAVGPU_OK;
}

int alloc_grid(navgpu_costmap* h, uint8_t** p, uint8_t value) {
  NAVGPU_CUDA(cudaMalloc(p, h->bytes()));
  NAVGPU_CUDA(cudaMemsetAsync(*p, value, h->bytes(), h->stream));
  return NAVGPU_OK;
}

// host mirror of Costmap2D::updateOrigin's scalar part (costmap_2d.cpp:264-275, 301-302); the cell shift runs on the
// device (k_shift_grid) into the other buffer of the ping-pong pair.
int roll_grid(navgpu_costmap* h, uint8_t* grid[2], int& cur, double& gox, double& goy, uint8_t def, double new_ox,
              double new_oy) {
  int cell_ox = int((new_ox - gox) / h->res), cell_oy = int((new_oy - goy) / h->res);
  double new_grid_ox = gox + cell_ox * h->res, new_grid_oy = goy + cell_oy * h->res;
  if (!grid[cur ^ 1]) NAVGPU_CUDA(cudaMalloc(&grid[cur ^ 1], h->bytes()));
  dim3 block(256), g((h->pitch + 255) / 256, h->sy);
  k_shift_grid<<<g, block, 0, h->stream>>>(grid[cur], grid[cur ^ 1], h->sx, h->sy, h->pitch, cell_ox, cell_oy, def);
  NAVGPU_LAUNCHED(1);
  cur ^= 1;
  gox = new_grid_ox;
  goy = new_grid_oy;
  return NAVGPU_OK;
}

int upload_tables(navgpu_costmap* h, Layer& L) {
  if (!L.tables_dirty) return NAVGPU_OK;
  const unsigned R = cell_distance(L.radius, h->res);
  build_tables(L.tables, R, h->res, L.inscribed, L.weight);
  if (L.mode == 0 && L.tables.ambiguous)
    return fail(NAVGPU_ERR_UNSUPPORTED, "inflation cost table is not a function of squared distance for R=%u", R);
  if (R > 254) return fail(NAVGPU_ERR_UNSUPPORTED, "cell inflation radius %u > 254", R);
  if (L.mode == 1) {
    if (R > 127) return fail(NAVGPU_ERR_UNSUPPORTED, "propagation mode carries sources as 8-bit offsets: R=%u > 127", R);
    for (uint16_t r : L.tables.rank)
      if (r != 0xffff && r > kPMaxRank) return fail(NAVGPU_ERR_UNSUPPORTED, "too many distinct distances for R=%u", R);
    const size_t n2 = L.tables.costs.size();
    if (n2 > L.table2d_capacity) {
      if (L.d_rank) cudaFree(L.d_rank);
      if (L.d_cost2d) cudaFree(L.d_cost2d);
      L.d_rank = nullptr; L.d_cost2d = nullptr;
      NAVGPU_CUDA(cudaMalloc(&L.d_rank, n2 * sizeof(uint16_t)));
      NAVGPU_CUDA(cudaMalloc(&L.d_cost2d, n2));
      L.table2d_capacity = n2;
    }
    NAVGPU_CUDA(cudaMemcpyAsync(L.d_rank, L.tables.rank.data(), n2 * sizeof(uint16_t), cudaMemcpyHostToDevice, h->stream));
    NAVGPU_CUDA(cudaMemcpyAsync(L.d_cost2d, L.tables.costs.data(), n2, cudaMemcpyHostToDevice, h->stream));
  }
  size_t n = L.tables.by_d2.size();
  if (n > L.cost_d2_capacity) {
    if (L.d_cost_d2) cudaFree(L.d_cost_d2);
    NAVGPU_CUDA(cudaMalloc(&L.d_cost_d2, n + 8));  // (k_inflate stages the table by 32-bit words)
    L.cost_d2_capacity = n;
  }
  NAVGPU_CUDA(cudaMemcpyAsync(L.d_cost_d2, L.tables.by_d2.data(), n, cudaMemcpyHostToDevice, h->stream));
  // the table lives in pageable host memory owned by this handle; make the copy complete before it can change
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  L.tables_dirty = false;
  return NAVGPU_OK;
}

// One sweep over the master grid: the two-kernel fast path (k_merge_seed [+ k_inflate], R <= 31) or the generic
// fused kernel (any R <= 254).  `seeds` is the handle's seed bitmask (sy x seed_pitch16(pitch) uint16, pads zero).
// everything inflation mode 1 needs besides the sweep's own arguments (buffers sized for the grid of the sweep)
struct PropBuffers {
  uint32_t* state = nullptr;
  uint32_t* list[2] = {nullptr, nullptr};
  PropCtl* ctl = nullptr;
  const uint16_t* rank = nullptr;
  const uint8_t* cost = nullptr;
  int max_blocks = 0;  // co-resident CTAs of k_inflate_propagate on this device
};

int propagate_max_blocks(int device, int R, int* out, size_t* smem_set) {
  const size_t smem = propagate_smem(R);
  if (smem > 200 * 1024) return fail(NAVGPU_ERR_UNSUPPORTED, "propagation tables for R=%d need %zu B of shared memory", R, smem);
  if (smem > *smem_set) {
    NAVGPU_CUDA(cudaFuncSetAttribute(k_inflate_propagate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    *smem_set = smem;
  }
  int per_sm = 0, sms = 0;
  NAVGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_inflate_propagate, kPThreads, smem));
  NAVGPU_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (per_sm < 1) return fail(NAVGPU_ERR_UNSUPPORTED, "k_inflate_propagate does not fit an SM for R=%d", R);
  *out = per_sm * sms;
  return NAVGPU_OK;
}

int launch_propagate(const UpdateArgs& a, const uint16_t* seeds, const PropBuffers& pb, cudaStream_t stream) {
  PropArgs pa;
  pa.master = a.master;
  pa.sx = a.sx; pa.sy = a.sy; pa.pitch = a.pitch;
  pa.win = a.win;
  pa.R = a.R;
  pa.seeds = reinterpret_cast<const uint32_t*>(seeds);
  pa.state = pb.state;
  pa.rank = pb.rank;
  pa.cost = pb.cost;
  pa.ctl = pb.ctl;
  pa.list[0] = pb.list[0];
  pa.list[1] = pb.list[1];
  // a small grid needs few CTAs (the per-round barrier is cheaper), a large one every co-resident CTA
  const long long cells = (long long)a.pitch * a.sy;
  const int blocks = (int)std::max<long long>(1, std::min<long long>(cells / 8192, pb.max_blocks));
  // barrier counters and list sizes 0, pending-rank slots "none"
  NAVGPU_CUDA(cudaMemsetAsync(pb.ctl, 0, sizeof(PropCtl), stream));
  NAVGPU_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(pb.ctl) + offsetof(PropCtl, kmin), 0xff, sizeof(pb.ctl->kmin), stream));
  void* args[] = {&pa};
  NAVGPU_CUDA(cudaLaunchCooperativeKernel((const void*)k_inflate_propagate, dim3(blocks), dim3(kPThreads), args,
                                          propagate_smem(a.R), stream));
  NAVGPU_LAUNCHED(1);
  return NAVGPU_OK;
}

struct TileFlags {  // early mode: k_merge_seed -> k_inflate per-tile hand-over (MergeSeedArgs::ready)
  unsigned* ready = nullptr;
  unsigned epoch = 0;
  unsigned* done = nullptr;        // InflateArgs::done
  bool* handed_over = nullptr;     // out: the sweep used the per-tile flags (and published `done`)
};
static_assert(kMirrorInflateTileW == kITX && kMirrorInflateTileH == kITY, "k_mirror_diff waits for k_inflate's tiles");

int launch_sweep(const UpdateArgs& a, uint16_t* seeds, cudaStream_t stream, bool force_generic, cudaEvent_t ev_mid = nullptr,
                 const PropBuffers* prop = nullptr, const TileFlags* flags = nullptr) {
  const int R = a.R;
  if ((R <= 31 && !force_generic) || (prop && R > 0)) {
    MergeSeedArgs m;
    m.master = a.master;
    m.sx = a.sx; m.sy = a.sy; m.pitch = a.pitch;
    m.def = a.def;
    m.do_reset = a.do_reset;
    m.win = a.win;
    m.ml = a.ml;
    m.R = R;
    m.seeds = seeds;
    m.early = a.early; m.ex0 = a.ex0; m.exn = a.exn; m.ey0 = a.ey0; m.eyn = a.eyn;
    m.obst_flag = a.obst_flag; m.obst_epoch = a.obst_epoch;
    m.lean = a.ml.n >= 1 && a.ml.n <= 2 && a.ml.policy[0] == NAVGPU_TRUE_OVERWRITE &&
             (a.ml.n == 1 || a.ml.policy[1] == NAVGPU_MAX || a.ml.policy[1] == NAVGPU_OVERWRITE);
    if (R > 0 && !seeds) return fail(NAVGPU_ERR_INVALID, "seed bitmask missing");
    dim3 block(kMSGroupsX, kMSRowsY);
    dim3 grid((a.pitch + kMSGroupsX * 16 - 1) / (kMSGroupsX * 16), (a.sy + kMSTileH - 1) / kMSTileH);
    const bool handover = flags && flags->ready && a.early && R > 0 && !(prop && R > 0) && !ev_mid;
    if (handover) { m.ready = flags->ready; m.epoch = flags->epoch; }
    if (a.ml.n > 0 || a.do_reset || R > 0) {
      NAVGPU_CUDA(launch_pdl(k_merge_seed, grid, block, 0, stream, m));
      NAVGPU_LAUNCHED(1);
    }
    if (ev_mid) cudaEventRecord(ev_mid, stream);
    if (prop && R > 0) return launch_propagate(a, seeds, *prop, stream);
    if (R > 0) {
      InflateArgs ia;
      ia.master = a.master;
      ia.sx = a.sx; ia.sy = a.sy; ia.pitch = a.pitch;
      ia.win = a.win;
      ia.R = R;
      ia.reach2 = a.reach2;
      ia.cost_d2 = a.cost_d2;
      ia.seeds = reinterpret_cast<const uint32_t*>(seeds);
      if (handover) {
        ia.ready = flags->ready; ia.epoch = flags->epoch; ia.ready_pitch = (int)grid.x;
        ia.done = flags->done;
        if (flags->handed_over) *flags->handed_over = flags->done != nullptr;
      }
      dim3 igrid((a.sx + kITX - 1) / kITX, (a.sy + kITY - 1) / kITY);
      // the instantiation whose unrolled row walk just covers the effective reach (what k_inflate calls R)
      const int reach = (int)sqrtf((float)a.reach2 + 0.5f);
      ia.reach = reach;
      if (reach <= 12) NAVGPU_CUDA(launch_pdl(k_inflate<12>, igrid, dim3(kIThreads), 0, stream, ia));
      else if (reach <= 20) NAVGPU_CUDA(launch_pdl(k_inflate<20>, igrid, dim3(kIThreads), 0, stream, ia));
      else NAVGPU_CUDA(launch_pdl(k_inflate<31>, igrid, dim3(kIThreads), 0, stream, ia));
      NAVGPU_LAUNCHED(1);
    }
    return NAVGPU_OK;
  }
  size_t smem = update_costs_smem(R);
  if (smem > 200 * 1024) return fail(NAVGPU_ERR_UNSUPPORTED, "cell inflation radius %d needs %zu B of shared memory", R, smem);
  if (smem > 48 * 1024)
    NAVGPU_CUDA(cudaFuncSetAttribute(k_update_costs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((a.sx + kTX - 1) / kTX, (a.sy + kTY - 1) / kTY);
  k_update_costs<<<grid, kUpdateThreads, smem, stream>>>(a);
  NAVGPU_LAUNCHED(1);
  return NAVGPU_OK;
}

int ensure_seeds(uint16_t** seeds, size_t* cap, unsigned pitch, unsigned sy, cudaStream_t stream) {
  const size_t need = size_t(seed_pitch16(pitch)) * sy * sizeof(uint16_t);
  if (*seeds && need <= *cap) return NAVGPU_OK;
  if (*seeds) cudaFree(*seeds);
  *seeds = nullptr;
  NAVGPU_CUDA(cudaMalloc(seeds, need));
  NAVGPU_CUDA(cudaMemsetAsync(*seeds, 0, need, stream));  // the pad groups stay zero for good
  *cap = need;
  return NAVGPU_OK;
}

int ensure_prop(navgpu_costmap* h, const Layer& L, PropBuffers* pb) {
  if (!h->d_prop_state) {  // per-cell state + the two frontier lists (a cell is listed at most once per list)
    NAVGPU_CUDA(cudaMalloc(&h->d_prop_state, 3 * h->bytes() * sizeof(uint32_t)));
    NAVGPU_CUDA(cudaMalloc(&h->d_prop_ctl, sizeof(PropCtl)));
  }
  NAVGPU_TRY(propagate_max_blocks(h->device, (int)L.tables.R, &h->prop_max_blocks, &h->prop_smem_set));
  pb->state = h->d_prop_state;
  pb->list[0] = h->d_prop_state + h->bytes();
  pb->list[1] = h->d_prop_state + 2 * h->bytes();
  pb->ctl = h->d_prop_ctl;
  pb->rank = L.d_rank;
  pb->cost = L.d_cost2d;
  pb->max_blocks = h->prop_max_blocks;
  return NAVGPU_OK;
}

struct EarlyBox {  // see UpdateArgs::early
  int on = 0, x0 = 0, xn = 0, y0 = 0, yn = 0;
  const unsigned* flag = nullptr;  // UpdateArgs::obst_flag
  unsigned epoch = 0;
};

int launch_update(navgpu_costmap* h, const MergeLayers& ml, int do_reset, int R, const uint8_t* cost_d2, int reach2 = 0,
                  const Layer* infl = nullptr, const EarlyBox* early = nullptr) {
  UpdateArgs a;
  a.early = early && early->on && do_reset ? 1 : 0;
  a.ex0 = early ? early->x0 : 0; a.exn = early ? early->xn : 0; a.ey0 = early ? early->y0 : 0; a.eyn = early ? early->yn : 0;
  if (a.early && early->flag) { a.obst_flag = early->flag; a.obst_epoch = early->epoch; }
  a.master = h->master[h->cur];
  a.sx = h->sx; a.sy = h->sy; a.pitch = h->pitch;
  a.def = h->def;
  a.do_reset = do_reset;
  a.win = h->d_win;
  a.ml = ml;
  a.R = R;
  a.cost_d2 = cost_d2;
  a.reach2 = reach2;
  PropBuffers pb;
  const bool propagate = infl && infl->mode == 1 && R > 0;
  if (propagate) NAVGPU_TRY(ensure_prop(h, *infl, &pb));
  if (R > 0 && (R <= 31 || propagate)) NAVGPU_TRY(ensure_seeds(&h->d_seeds, &h->seeds_capacity, h->pitch, h->sy, h->stream));
  if (h->profile && R > 0) cudaEventRecord(h->ev_sweep[0], h->stream);
  TileFlags tf;
  if (a.early && R > 0 && R <= 31 && !propagate) {
    const size_t n_tiles = size_t((a.pitch + kMSGroupsX * 16 - 1) / (kMSGroupsX * 16)) * ((a.sy + kMSTileH - 1) / kMSTileH);
    if (!h->d_tile_ready) {
      NAVGPU_CUDA(cudaMalloc(&h->d_tile_ready, n_tiles * sizeof(unsigned)));
      NAVGPU_CUDA(cudaMemsetAsync(h->d_tile_ready, 0, n_tiles * sizeof(unsigned), h->stream));
    }
    tf.ready = h->d_tile_ready;
    tf.epoch = ++h->sweep_epoch;
    const size_t n_itiles = size_t((a.sx + kITX - 1) / kITX) * ((a.sy + kITY - 1) / kITY);
    if (n_itiles > h->inflate_done_capacity) {
      if (h->d_inflate_done) cudaFree(h->d_inflate_done);
      NAVGPU_CUDA(cudaMalloc(&h->d_inflate_done, n_itiles * sizeof(unsigned)));
      NAVGPU_CUDA(cudaMemsetAsync(h->d_inflate_done, 0, n_itiles * sizeof(unsigned), h->stream));
      h->inflate_done_capacity = n_itiles;
    }
    tf.done = h->d_inflate_done;
  }
  bool handed_over = false;
  tf.handed_over = &handed_over;
  h->inflate_done_epoch = 0;  // (whatever sweep ran before is no longer the last one)
  NAVGPU_TRY(launch_sweep(a, h->d_seeds, h->stream, h->force_generic, h->profile && R > 0 ? h->ev_mid : nullptr,
                          propagate ? &pb : nullptr, &tf));
  if (h->profile && R > 0) cudaEventRecord(h->ev_sweep[1], h->stream);
  if (handed_over) {
    h->inflate_done_epoch = tf.epoch;
    h->inflate_done_pitch = (int)((a.sx + kITX - 1) / kITX);
  }
  return NAVGPU_OK;
}

// Host part of ObstacleLayer::updateCosts' footprint clearing (obstacle_layer.cpp:432-435 -> setConvexPolygonCost,
// costmap_2d.cpp:315-342): vertices to cells; *mode = 0 nothing to clear, 1 fits k_obstacle_update, 2 stand-alone kernel
int footprint_polygon(navgpu_costmap* h, const Layer& L, PolyArgs& pa, int* mode) {
  *mode = 0;
  pa.n = 0;
  if (L.transformed_footprint.size() > 32) return fail(NAVGPU_ERR_UNSUPPORTED, "footprint with more than 32 vertices");
  for (const Pt& p : L.transformed_footprint) {  // worldToMap, costmap_2d.cpp:208-220; any vertex off the map: no clearing
    if (p.x < L.ox || p.y < L.oy) return NAVGPU_OK;
    unsigned mx = (int)((p.x - L.ox) / h->res), my = (int)((p.y - L.oy) / h->res);
    if (!(mx < h->sx && my < h->sy)) return NAVGPU_OK;
    pa.vx[pa.n] = (int)mx;
    pa.vy[pa.n] = (int)my;
    ++pa.n;
  }
  if (pa.n < 3) return NAVGPU_OK;
  long long outline = 0, minx = pa.vx[0], maxx = pa.vx[0], miny = pa.vy[0], maxy = pa.vy[0];
  for (int k = 0; k < pa.n; ++k) {
    int k1 = (k + 1) % pa.n;
    outline += std::max(std::abs(pa.vx[k1] - pa.vx[k]), std::abs(pa.vy[k1] - pa.vy[k])) + 1;
    minx = std::min<long long>(minx, pa.vx[k]); maxx = std::max<long long>(maxx, pa.vx[k]);
    miny = std::min<long long>(miny, pa.vy[k]); maxy = std::max<long long>(maxy, pa.vy[k]);
  }
  const long long cells = outline + (maxx - minx + 1) * (maxy - miny + 1);
  if (cells > kPolyMaxCells || h->sx > 65535 || h->sy > 65535)
    return fail(NAVGPU_ERR_UNSUPPORTED, "footprint polygon covers too many cells for the device rasteriser");
  *mode = cells <= kPolySmallCells ? 1 : 2;
  return NAVGPU_OK;
}

// One LayeredCostmap::updateMap cycle (layered_costmap.cpp:79-150), enqueued on the handle's stream.
int enqueue_update(navgpu_costmap* h, double rx, double ry, double ryaw) {
  NAVGPU_TRY(use_device(h));
  // The inflation tables first: a radius the sweeps cannot run is refused before the cycle changes anything, so the
  // handle stays as it was -- grid layer updates and reinflation requests still pending, layer grids and the host
  // mirror's bookkeeping untouched -- and the next accepted configuration picks up where it left off.
  for (Layer& L : h->layers)
    if (L.kind == 2 && L.enabled) NAVGPU_TRY(upload_tables(h, L));
  // rolling window: master origin follows the robot (:86-91)
  if (h->rolling)
    NAVGPU_TRY(roll_grid(h, h->master, h->cur, h->ox, h->oy, h->def, rx - h->size_m_x() / 2, ry - h->size_m_y() / 2));
  if (h->layers.empty()) return NAVGPU_OK;

  // ---- updateBounds of every plugin, in order (:96-115): host-side scalars first
  BoundsArgs ba;
  ba.n_layers = (int)h->layers.size();
  ba.master = h->geom(h->ox, h->oy);
  unsigned max_cell_radius = 0;
  for (const Layer& L : h->layers)
    if (L.kind == 2) max_cell_radius = std::max(max_cell_radius, cell_distance(L.radius, h->res));
  ba.mirror_dirty = h->d_mirror_dirty;
  ba.mirror_pad = 2 * (int)max_cell_radius + 2;
  if (h->rolling) {  // the grid may shift under the shadow
    h->mirror_all = true;
    h->master_clean = false;
  }
  int last_obstacle = -1;
  // Is this cycle's window the whole map as far as the host can tell (a grid layer updated as a whole, an inflation
  // layer that must re-inflate), and where can the obstacle kernels write?  Then the merge sweep need not wait for them
  // outside that box (UpdateArgs::early).
  bool whole_map = false, box_known = !h->rolling;
  double ebx0 = 1e300, eby0 = 1e300, ebx1 = -1e300, eby1 = -1e300;
  for (size_t li = 0; li < h->layers.size(); ++li) {
    Layer& L = h->layers[li];
    BoundsLayer& B = ba.layer[li];
    B.kind = L.kind == 2 ? 2 : 0;
    B.flag = 0;
    B.hx0 = B.hy0 = B.hx1 = B.hy1 = 0;
    if (L.kind == 0) {  // StaticLayer::updateBounds, non-rolling semantics (static_layer.cpp:263-285)
      if (!h->rolling && !L.updated) continue;
      B.flag = 1;
      B.hx0 = L.ox + (L.ux + 0.5) * h->res;  // mapToWorld, costmap_2d.cpp:202-206
      B.hy0 = L.oy + (L.uy + 0.5) * h->res;
      B.hx1 = L.ox + (L.ux + L.uw + 0.5) * h->res;
      B.hy1 = L.oy + (L.uy + L.uh + 0.5) * h->res;
      if (L.ux == 0 && L.uy == 0 && L.uw >= h->sx && L.uh >= h->sy && L.ox == h->ox && L.oy == h->oy) whole_map = true;
      L.updated = false;
    } else if (L.kind == 1) {  // ObstacleLayer::updateBounds (obstacle_layer.cpp:340-413)
      if (h->rolling) {
        if (L.voxel) {  // VoxelLayer::updateOrigin moves the columns with the 2-D cells (voxel_layer.cpp:371-438)
          const double new_ox = rx - h->size_m_x() / 2, new_oy = ry - h->size_m_y() / 2;
          const int cell_ox = int((new_ox - L.ox) / h->res), cell_oy = int((new_oy - L.oy) / h->res);
          if (!L.vox[L.cur ^ 1]) NAVGPU_CUDA(cudaMalloc(&L.vox[L.cur ^ 1], h->bytes() * sizeof(uint32_t)));
          dim3 block(256), g((h->pitch + 255) / 256, h->sy);
          k_shift_voxels<<<g, block, 0, h->stream>>>(L.vox[L.cur], L.vox[L.cur ^ 1], h->sx, h->sy, h->pitch, cell_ox, cell_oy);
          NAVGPU_LAUNCHED(1);
        }
        NAVGPU_TRY(roll_grid(h, L.grid, L.cur, L.ox, L.oy, L.def, rx - h->size_m_x() / 2, ry - h->size_m_y() / 2));
      }
      L.transformed_footprint.clear();
      if (!L.enabled) continue;
      last_obstacle = (int)li;
      double bx0 = 1e300, by0 = 1e300, bx1 = -1e300, by1 = -1e300;
      // raytraceFreespace touches the sensor origin once per clearing observation whose origin is on the map
      // (:504-521); origins and geometry are host-side scalars, the per-ray end points are touched on the device
      for (const HostObs& o : L.obs) {
        if (!o.clearing || L.voxel) continue;  // VoxelLayer::raytraceFreespace does not touch the sensor origin
        if (o.ox < L.ox || o.oy < L.oy) continue;
        unsigned mx = (int)((o.ox - L.ox) / h->res), my = (int)((o.oy - L.oy) / h->res);
        if (!(mx < h->sx && my < h->sy)) continue;
        bx0 = std::min(o.ox, bx0); by0 = std::min(o.oy, by0);
        bx1 = std::max(o.ox, bx1); by1 = std::max(o.oy, by1);
      }
      if (L.footprint_clearing) {  // updateFootprint (:415-425) with transformFootprint (footprint.cpp:106-120)
        double cos_th = cos(ryaw), sin_th = sin(ryaw);
        for (const Pt& p : h->footprint)
          L.transformed_footprint.push_back(Pt{rx + (p.x * cos_th - p.y * sin_th), ry + (p.x * sin_th + p.y * cos_th)});
        for (const Pt& p : L.transformed_footprint) {
          bx0 = std::min(p.x, bx0); by0 = std::min(p.y, by0);
          bx1 = std::max(p.x, bx1); by1 = std::max(p.y, by1);
        }
      }
      if (bx1 >= bx0) {
        B.flag = 1;
        B.hx0 = bx0; B.hy0 = by0; B.hx1 = bx1; B.hy1 = by1;
      }
      if (L.voxel || !L.touch_box_valid || L.ox != h->ox || L.oy != h->oy) box_known = false;
      if (L.tbx1 >= L.tbx0 && L.tby1 >= L.tby0) {
        ebx0 = std::min(ebx0, L.tbx0); eby0 = std::min(eby0, L.tby0);
        ebx1 = std::max(ebx1, L.tbx1); eby1 = std::max(eby1, L.tby1);
      }
      for (const Pt& p : L.transformed_footprint) {
        ebx0 = std::min(ebx0, p.x); eby0 = std::min(eby0, p.y);
        ebx1 = std::max(ebx1, p.x); eby1 = std::max(eby1, p.y);
      }
    } else {  // InflationLayer::updateBounds runs on the device (needs the device-accumulated bounds)
      if (L.need_reinflation) whole_map = true;
      B.flag = L.need_reinflation ? 1 : 0;
      B.hx0 = L.radius;
      L.need_reinflation = false;
    }
  }

  EarlyBox early;
  if (whole_map && box_known) {
    early.on = 1;
    if (ebx1 >= ebx0 && eby1 >= eby0) {  // cells, two to spare on every side, clamped to the map
      auto cell = [&](double w, double origin, int size, int pad) {
        const double c = std::floor((w - origin) / h->res) + pad;
        return (int)std::min<double>(size, std::max(0.0, c));
      };
      early.x0 = cell(ebx0, h->ox, (int)h->sx, -2); early.xn = cell(ebx1, h->ox, (int)h->sx, 3);
      early.y0 = cell(eby0, h->oy, (int)h->sy, -2); early.yn = cell(eby1, h->oy, (int)h->sy, 3);
    }
  }
  // ---- device part: one k_obstacle_update per enabled obstacle layer (ray-trace clearing, then marking, then the
  // footprint polygon of updateCosts); the last one also finalises the bounds into the cycle's window
  bool standalone_polygon = false;  // a k_polygon_clear launch follows some obstacle kernel: no early "grids done" flag
  for (size_t li = 0; li < h->layers.size(); ++li) {
    Layer& L = h->layers[li];
    if (L.kind != 1 || !L.enabled) continue;
    if (L.voxel) {
      VoxelArgs va;
      va.grid = L.grid[L.cur];
      va.vox = L.vox[L.cur];
      va.g = h->geom(L.ox, L.oy);
      va.v = L.vg;
      va.clear = L.d_clear; va.mark = L.d_mark; va.xyz = L.d_xyz;
      va.n_clear = L.n_clear; va.total_rays = L.total_rays; va.n_mark = L.n_mark; va.total_marks = L.total_marks;
      va.max_obstacle_height = L.max_obstacle_height;
      va.box = h->d_boxes + li;
      va.mark_cells = L.d_mark_cells;
      va.ticket = h->d_ticket;
      int vmode = 0;
      if (L.footprint_clearing) NAVGPU_TRY(footprint_polygon(h, L, va.poly, &vmode));
      va.do_poly = vmode == 1;
      va.do_finalize = (int)li == last_obstacle;
      if (va.do_finalize) va.ba = ba;
      va.boxes = h->d_boxes; va.infl = h->d_infl; va.win = h->d_win;
      const int vblocks = std::max(1, (L.total_rays * 32 + kObstacleThreads - 1) / kObstacleThreads);
      k_voxel_clear<<<vblocks, kObstacleThreads, 0, h->stream>>>(va);
      k_voxel_commit<<<vblocks, kObstacleThreads, 0, h->stream>>>(va);
      NAVGPU_LAUNCHED(2);
      if (vmode == 2) {
        size_t smem = 2 * kPolyMaxCells * sizeof(uint32_t);
        if (!h->poly_attr_set) {
          NAVGPU_CUDA(cudaFuncSetAttribute(k_polygon_clear, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
          h->poly_attr_set = true;
        }
        k_polygon_clear<<<1, 256, smem, h->stream>>>(L.grid[L.cur], h->pitch, va.poly, kFree);
        NAVGPU_LAUNCHED(1);
      }
      continue;
    }
    ObstacleArgs oa;
    oa.grid = L.grid[L.cur];
    oa.g = h->geom(L.ox, L.oy);
    oa.clear = L.d_clear; oa.mark = L.d_mark; oa.xyz = L.d_xyz;
    if (L.n_clear <= kInlineObs) std::copy(L.h_clear.begin(), L.h_clear.end(), oa.clear_inline);
    if (L.n_mark <= kInlineObs) std::copy(L.h_mark.begin(), L.h_mark.end(), oa.mark_inline);
    oa.n_clear = L.n_clear; oa.total_rays = L.total_rays; oa.n_mark = L.n_mark; oa.total_marks = L.total_marks;
    oa.max_obstacle_height = L.max_obstacle_height;
    oa.box = h->d_boxes + li;
    oa.mark_cells = L.d_mark_cells;
    oa.ticket = h->d_ticket;
    int mode = 0;
    if (L.footprint_clearing) NAVGPU_TRY(footprint_polygon(h, L, oa.poly, &mode));
    oa.do_poly = mode == 1;
    oa.do_finalize = (int)li == last_obstacle;
    if (oa.do_finalize) oa.ba = ba;
    oa.tile_used = L.d_tile_used;
    if (mode == 2) standalone_polygon = true;
    if (early.on && (int)li == last_obstacle && !standalone_polygon) {
      oa.done_flag = h->d_obst_done;
      oa.done_epoch = ++h->obst_epoch;
      early.flag = h->d_obst_done;
      early.epoch = oa.done_epoch;
    }
    oa.boxes = h->d_boxes; oa.infl = h->d_infl; oa.win = h->d_win;
    const int blocks = std::max(1, (L.total_rays + kObstacleRayWarps - 1) / kObstacleRayWarps);
    k_obstacle_update<<<blocks, kObstacleUpdateThreads, 0, h->stream>>>(oa);
    NAVGPU_LAUNCHED(1);
    if (mode == 2) {  // large footprint: stand-alone rasteriser with dynamic shared memory
      size_t smem = 2 * kPolyMaxCells * sizeof(uint32_t);
      if (!h->poly_attr_set) {
        NAVGPU_CUDA(cudaFuncSetAttribute(k_polygon_clear, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        h->poly_attr_set = true;
      }
      k_polygon_clear<<<1, 256, smem, h->stream>>>(L.grid[L.cur], h->pitch, oa.poly, kFree);
      NAVGPU_LAUNCHED(1);
    }
  }
  if (last_obstacle < 0) {
    k_finalize_bounds<<<1, 32, 0, h->stream>>>(ba, h->d_boxes, h->d_infl, h->d_win);
    NAVGPU_LAUNCHED(1);
  }

  // ---- resetMap + updateCosts of every plugin, in order (:137-142), fused into as few sweeps as possible:
  // consecutive cost layers merge in one pass, an inflation layer closes the pass.
  // host mirror: a whole-map cycle on a grid that was a pure function of the layers, with layers that changed only inside
  // the obstacle kernels' box, changes master cells only within that box grown by the inflation radius
  if (early.on && h->master_clean && !h->content_changed) {
    if (early.xn > early.x0 && early.yn > early.y0) {
      const int pad = (int)max_cell_radius + 1;
      const int x0 = std::max(0, early.x0 - pad), xn = std::min((int)h->sx, early.xn + pad);
      const int y0 = std::max(0, early.y0 - pad), yn = std::min((int)h->sy, early.yn + pad);
      if (h->refine[1] > h->refine[0]) {
        h->refine[0] = std::min(h->refine[0], x0); h->refine[1] = std::max(h->refine[1], xn);
        h->refine[2] = std::min(h->refine[2], y0); h->refine[3] = std::max(h->refine[3], yn);
      } else {
        h->refine[0] = x0; h->refine[1] = xn; h->refine[2] = y0; h->refine[3] = yn;
      }
    }
  } else {
    h->refine_valid = false;
  }
  h->master_clean = whole_map && !h->rolling;
  h->content_changed = false;
  MergeLayers ml;
  ml.n = 0;
  int do_reset = 1;
  bool pending = true;  // the reset itself must happen even with no enabled layer
  for (size_t li = 0; li < h->layers.size(); ++li) {
    Layer& L = h->layers[li];
    if (L.kind == 0 || L.kind == 1) {
      if (!L.enabled) continue;
      int policy = L.kind == 0 ? L.policy
                               : (L.combination_method == 0 ? NAVGPU_OVERWRITE
                                                            : (L.combination_method == 1 ? NAVGPU_MAX : NAVGPU_NOTHING));
      if (policy == NAVGPU_NOTHING) continue;
      ml.grid[ml.n] = L.grid[L.cur];
      ml.policy[ml.n] = policy;
      ml.used[ml.n] = L.d_tile_used;
      ++ml.n;
      pending = true;
    } else {
      if (!L.enabled) continue;  // (its tables were uploaded at the start of the cycle)
      if (L.tables.R == 0) continue;  // the reference dereferences NULL tables here; we make it a no-op
      if (!do_reset && ml.n > 0) {    // merges that read what a previous inflation wrote: keep them a separate pass
        NAVGPU_TRY(launch_update(h, ml, 0, 0, nullptr));
        ml.n = 0;
      }
      NAVGPU_TRY(launch_update(h, ml, do_reset, (int)L.tables.R, L.d_cost_d2, L.tables.reach2, &L, &early));
      ml.n = 0;
      do_reset = 0;
      pending = false;
    }
  }
  if (pending) NAVGPU_TRY(launch_update(h, ml, do_reset, 0, nullptr, 0, nullptr, &early));
  return NAVGPU_OK;
}

}  // namespace

extern "C" {

const char* navgpu_last_error(void) { return last_error_ref().c_str(); }

int navgpu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

uint64_t navgpu_launch_count(void) { return launch_counter().load(); }

int navgpu_costmap_create(navgpu_costmap** out, uint32_t size_x, uint32_t size_y, double resolution, double origin_x,
                          double origin_y, int rolling_window, int track_unknown, int device) {
  if (!out || size_x == 0 || size_y == 0 || !(resolution > 0)) return fail(NAVGPU_ERR_INVALID, "bad costmap geometry");
  if (navgpu_device_count() <= device) return fail(NAVGPU_ERR_CUDA, "no CUDA device %d (libnavgpu has no CPU fallback)", device);
  std::unique_ptr<navgpu_costmap> h(new navgpu_costmap);
  h->device = device;
  NAVGPU_CUDA(cudaSetDevice(device));
  NAVGPU_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  h->sx = size_x; h->sy = size_y; h->pitch = grid_pitch(size_x);
  h->res = resolution; h->ox = origin_x; h->oy = origin_y;
  h->rolling = rolling_window != 0;
  h->track_unknown = track_unknown != 0;
  h->def = track_unknown ? kNoInfo : kFree;  // layered_costmap.cpp:53-56
  NAVGPU_TRY(alloc_grid(h.get(), &h->master[0], h->def));
  NAVGPU_CUDA(cudaMalloc(&h->d_boxes, sizeof(DevBox) * kMaxLayers));
  NAVGPU_CUDA(cudaMalloc(&h->d_infl, sizeof(InflationBoundsState) * kMaxLayers));
  NAVGPU_CUDA(cudaMalloc(&h->d_win, sizeof(DevWindow)));
  NAVGPU_CUDA(cudaMalloc(&h->d_ticket, sizeof(unsigned)));
  NAVGPU_CUDA(cudaMemset(h->d_ticket, 0, sizeof(unsigned)));
  {
    // One L1 / shared-memory split (the largest shared-memory carve-out, which k_inflate's 8 x 27 KB need anyway) for the
    // three kernels of a cycle: CTAs of two kernels share an SM only if its split suits both, and an SM must drain to
    // change it.  With the same split k_inflate's CTAs move in as k_merge_seed's leave instead of waiting for the SM to
    // empty -- also on the SMs that hold the merge CTAs waiting for the obstacle kernel, or that kernel's last CTA.
    // (k_merge_seed streams and k_obstacle_update scatters single bytes: neither misses the L1 it gives up.)
    static bool done_for_device[64] = {};
    if (h->device >= 0 && h->device < 64 && !done_for_device[h->device]) {
      done_for_device[h->device] = true;
      const int c = cudaSharedmemCarveoutMaxShared;
      NAVGPU_CUDA(cudaFuncSetAttribute(k_obstacle_update, cudaFuncAttributePreferredSharedMemoryCarveout, c));
      NAVGPU_CUDA(cudaFuncSetAttribute(k_merge_seed, cudaFuncAttributePreferredSharedMemoryCarveout, c));
      NAVGPU_CUDA(cudaFuncSetAttribute(k_inflate<12>, cudaFuncAttributePreferredSharedMemoryCarveout, c));
      NAVGPU_CUDA(cudaFuncSetAttribute(k_inflate<20>, cudaFuncAttributePreferredSharedMemoryCarveout, c));
      NAVGPU_CUDA(cudaFuncSetAttribute(k_inflate<31>, cudaFuncAttributePreferredSharedMemoryCarveout, c));
      NAVGPU_CUDA(cudaFuncSetAttribute(k_mirror_diff, cudaFuncAttributePreferredSharedMemoryCarveout, c));
    }
  }
  NAVGPU_CUDA(cudaMalloc(&h->d_obst_done, sizeof(unsigned)));
  NAVGPU_CUDA(cudaMemset(h->d_obst_done, 0, sizeof(unsigned)));
  NAVGPU_CUDA(cudaMallocHost(&h->h_win, sizeof(DevWindow)));
  DevBox boxes[kMaxLayers];
  InflationBoundsState infl[kMaxLayers];
  for (int i = 0; i < kMaxLayers; ++i) {
    boxes[i] = DevBox{~0ull, ~0ull, 0ull, 0ull};
    const double fm = std::numeric_limits<float>::max();  // inflation_layer.cpp:63-66
    infl[i] = InflationBoundsState{-fm, -fm, fm, fm};
  }
  NAVGPU_CUDA(cudaMemcpy(h->d_boxes, boxes, sizeof(boxes), cudaMemcpyHostToDevice));
  NAVGPU_CUDA(cudaMemcpy(h->d_infl, infl, sizeof(infl), cudaMemcpyHostToDevice));
  NAVGPU_CUDA(cudaMemset(h->d_win, 0, sizeof(DevWindow)));
  NAVGPU_CUDA(cudaMalloc(&h->d_mirror_dirty, sizeof(DevWindow)));
  NAVGPU_CUDA(cudaMemset(h->d_mirror_dirty, 0, sizeof(DevWindow)));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  *out = h.release();
  return NAVGPU_OK;
}

int navgpu_costmap_destroy(navgpu_costmap* h) {
  if (!h) return NAVGPU_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (Layer& L : h->layers) {
    cudaFree(L.grid[0]); cudaFree(L.grid[1]);
    cudaFree(L.d_clear); cudaFree(L.d_mark); cudaFree(L.d_xyz); cudaFree(L.d_cost_d2); cudaFree(L.d_rank); cudaFree(L.d_cost2d); cudaFree(L.d_mark_cells); cudaFree(L.d_scan);
    if (L.h_stage) cudaFreeHost(L.h_stage);
    if (L.ev_stage) cudaEventDestroy(L.ev_stage);
    cudaFree(L.vox[0]); cudaFree(L.vox[1]); cudaFree(L.d_tile_used);
  }
  cudaFree(h->master[0]); cudaFree(h->master[1]);
  cudaFree(h->d_boxes); cudaFree(h->d_infl); cudaFree(h->d_win); cudaFree(h->d_seeds); cudaFree(h->d_ticket); cudaFree(h->d_obst_done); cudaFree(h->d_inflate_done); cudaFree(h->d_occupancy);
  cudaFree(h->d_prop_state); cudaFree(h->d_prop_ctl);
  cudaFree(h->d_shadow); cudaFree(h->d_mirror_counters); cudaFree(h->d_mirror_dirty); cudaFree(h->d_tile_ready);
  if (h->h_mirror_stage) cudaFreeHost(h->h_mirror_stage);
  if (h->h_mirror_tiles) cudaFreeHost(h->h_mirror_tiles);
  if (h->h_mirror_ctl) cudaFreeHost(h->h_mirror_ctl);
  cudaFreeHost(h->h_win);
  cudaStreamDestroy(h->stream);
  delete h;
  return NAVGPU_OK;
}

static int add_cost_layer(navgpu_costmap* h, Layer& L) {
  h->content_changed = true;
  // CostmapLayer::matchSize (costmap_layer.cpp:14-19): same geometry as the master, filled with the default value
  L.def = h->track_unknown ? kNoInfo : kFree;
  L.ox = h->ox;
  L.oy = h->oy;
  NAVGPU_TRY(alloc_grid(h, &L.grid[0], L.def));
  return NAVGPU_OK;
}

int navgpu_costmap_add_grid_layer(navgpu_costmap* h, int policy, int* layer_out) {
  if (!h || policy < 0 || policy > NAVGPU_NOTHING) return fail(NAVGPU_ERR_INVALID, "bad grid layer arguments");
  if (h->layers.size() >= (size_t)kMaxLayers) return fail(NAVGPU_ERR_UNSUPPORTED, "more than %d layers", kMaxLayers);
  NAVGPU_TRY(use_device(h));
  Layer L;
  L.kind = 0;
  L.policy = policy;
  NAVGPU_TRY(add_cost_layer(h, L));
  h->layers.push_back(L);
  if (layer_out) *layer_out = (int)h->layers.size() - 1;
  return NAVGPU_OK;
}

int navgpu_costmap_add_obstacle_layer(navgpu_costmap* h, int combination_method, int footprint_clearing,
                                      double max_obstacle_height, int* layer_out) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (h->layers.size() >= (size_t)kMaxLayers) return fail(NAVGPU_ERR_UNSUPPORTED, "more than %d layers", kMaxLayers);
  NAVGPU_TRY(use_device(h));
  Layer L;
  L.kind = 1;
  L.combination_method = combination_method;
  L.footprint_clearing = footprint_clearing != 0;
  L.max_obstacle_height = max_obstacle_height;
  NAVGPU_TRY(add_cost_layer(h, L));
  // The only writers of such a layer's grid are its own kernel's clears (FREE_SPACE) and marks: the tiles without a mark
  // are known to hold the default value.  Not for rolling maps (the grid shifts) or NO_INFORMATION defaults.
  if (!h->rolling && L.def == kFree) {
    const size_t n_tiles = size_t((h->pitch + kMarkTileW - 1) / kMarkTileW) * ((h->sy + kMarkTileH - 1) / kMarkTileH);
    NAVGPU_CUDA(cudaMalloc(&L.d_tile_used, n_tiles));
    NAVGPU_CUDA(cudaMemsetAsync(L.d_tile_used, 0, n_tiles, h->stream));
  }
  h->layers.push_back(L);
  if (layer_out) *layer_out = (int)h->layers.size() - 1;
  return NAVGPU_OK;
}

int navgpu_costmap_add_voxel_layer(navgpu_costmap* h, int combination_method, int footprint_clearing,
                                   double max_obstacle_height, double origin_z, double z_resolution, int z_voxels,
                                   int unknown_threshold, int mark_threshold, int* layer_out) {
  if (!h || z_voxels < 0 || z_voxels > 16 || !(z_resolution > 0) || unknown_threshold < 0 || mark_threshold < 0)
    return fail(NAVGPU_ERR_INVALID, "bad voxel layer arguments");
  if (mark_threshold != 0)  // with a positive threshold the reference's bounds depend on the order of the cloud points
    return fail(NAVGPU_ERR_UNSUPPORTED, "mark_threshold %d: only the reference's default 0 is implemented", mark_threshold);
  if (h->layers.size() >= (size_t)kMaxLayers) return fail(NAVGPU_ERR_UNSUPPORTED, "more than %d layers", kMaxLayers);
  NAVGPU_TRY(use_device(h));
  Layer L;
  L.kind = 1;
  L.voxel = true;
  L.combination_method = combination_method;
  L.footprint_clearing = footprint_clearing != 0;
  L.max_obstacle_height = max_obstacle_height;
  // VoxelLayer::reconfigureCB (voxel_layer.cpp:84-95): unknown_threshold_ = config.unknown_threshold + (16 - z_voxels)
  L.vg = VoxelGeom{origin_z, z_resolution, (unsigned)z_voxels, (unsigned)(unknown_threshold + (16 - z_voxels)), (unsigned)mark_threshold};
  NAVGPU_TRY(add_cost_layer(h, L));
  // VoxelGrid starts (and resets to) all-unknown columns (voxel_grid.cpp:41-59)
  NAVGPU_CUDA(cudaMalloc(&L.vox[0], h->bytes() * sizeof(uint32_t)));
  {
    std::vector<uint32_t> unknown(h->bytes(), 0x0000ffffu);
    NAVGPU_CUDA(cudaMemcpy(L.vox[0], unknown.data(), unknown.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  }
  h->layers.push_back(L);
  if (layer_out) *layer_out = (int)h->layers.size() - 1;
  return NAVGPU_OK;
}

int navgpu_layer_get_voxels(navgpu_costmap* h, int layer, uint32_t* host_out) {
  Layer* L = (h && layer >= 0 && layer < (int)h->layers.size()) ? &h->layers[layer] : nullptr;
  if (!L || !L->voxel || !host_out) return fail(NAVGPU_ERR_INVALID, "not a voxel layer");
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaMemcpy2DAsync(host_out, h->sx * sizeof(uint32_t), L->vox[L->cur], h->pitch * sizeof(uint32_t),
                                h->sx * sizeof(uint32_t), h->sy, cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

int navgpu_costmap_add_inflation_layer(navgpu_costmap* h, double inflation_radius, double cost_scaling_factor,
                                       int* layer_out) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (h->layers.size() >= (size_t)kMaxLayers) return fail(NAVGPU_ERR_UNSUPPORTED, "more than %d layers", kMaxLayers);
  Layer L;
  L.kind = 2;
  // onInitialize: the dynamic_reconfigure server first delivers the defaults (0.55, 10), which differ from the
  // constructor's zeros and therefore set need_reinflation_ (inflation_layer.cpp:71-108, 356-370)
  L.radius = inflation_radius;
  L.weight = cost_scaling_factor;
  L.inscribed = h->inscribed;
  L.need_reinflation = true;
  L.tables_dirty = true;
  h->layers.push_back(L);
  if (layer_out) *layer_out = (int)h->layers.size() - 1;
  return NAVGPU_OK;
}

int navgpu_costmap_set_footprint(navgpu_costmap* h, const double* xy, int n) {  // layered_costmap.cpp:163-173
  if (!h || n < 0 || (n > 0 && !xy)) return fail(NAVGPU_ERR_INVALID, "bad footprint");
  h->content_changed = true;
  h->footprint.clear();
  for (int i = 0; i < n; ++i) h->footprint.push_back(Pt{xy[2 * i], xy[2 * i + 1]});
  footprint_radii(h->footprint, h->inscribed, h->circumscribed);
  for (Layer& L : h->layers)
    if (L.kind == 2) {  // InflationLayer::onFootprintChanged (:160-170)
      L.inscribed = h->inscribed;
      L.need_reinflation = true;
      L.tables_dirty = true;
    }
  return NAVGPU_OK;
}

static Layer* get_layer(navgpu_costmap* h, int layer, int kind) {
  if (!h || layer < 0 || layer >= (int)h->layers.size()) return nullptr;
  Layer* L = &h->layers[layer];
  if (kind >= 0 && L->kind != kind) return nullptr;
  return L;
}

static void mark_whole(navgpu_costmap* h, Layer* L) {
  h->content_changed = true;  // (navgpu_grid_layer_set*: the layer's cells changed, not just its "updated" box)
  L->ux = L->uy = 0;
  L->uw = h->sx;
  L->uh = h->sy;
  L->updated = true;
}

int navgpu_grid_layer_set(navgpu_costmap* h, int layer, const uint8_t* host_data) {
  Layer* L = get_layer(h, layer, 0);
  if (!L || !host_data) return fail(NAVGPU_ERR_INVALID, "bad grid layer");
  h->content_changed = true;
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaMemcpy2DAsync(L->grid[L->cur], h->pitch, host_data, h->sx, h->sx, h->sy, cudaMemcpyHostToDevice, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  mark_whole(h, L);
  return NAVGPU_OK;
}

int navgpu_grid_layer_set_device(navgpu_costmap* h, int layer, const uint8_t* dev_data, uint32_t pitch) {
  Layer* L = get_layer(h, layer, 0);
  if (!L || !dev_data || pitch < h->sx) return fail(NAVGPU_ERR_INVALID, "bad grid layer");
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaMemcpy2DAsync(L->grid[L->cur], h->pitch, dev_data, pitch, h->sx, h->sy, cudaMemcpyDeviceToDevice, h->stream));
  mark_whole(h, L);
  return NAVGPU_OK;
}

int navgpu_grid_layer_set_occupancy(navgpu_costmap* h, int layer, const int8_t* host_occupancy, int track_unknown,
                                    uint8_t unknown_cost_value, uint8_t lethal_threshold, int trinary) {
  Layer* L = get_layer(h, layer, 0);
  if (!L || !host_occupancy) return fail(NAVGPU_ERR_INVALID, "bad grid layer");
  NAVGPU_TRY(use_device(h));
  int8_t* d_occ = nullptr;
  size_t n = size_t(h->sx) * h->sy;
  NAVGPU_CUDA(cudaMallocAsync(&d_occ, n, h->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(d_occ, host_occupancy, n, cudaMemcpyHostToDevice, h->stream));
  dim3 block(256), grid((h->sx + 255) / 256, h->sy);
  k_interpret_occupancy<<<grid, block, 0, h->stream>>>(d_occ, L->grid[L->cur], h->sx, h->sy, h->pitch, track_unknown,
                                                       unknown_cost_value, lethal_threshold, trinary);
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaFreeAsync(d_occ, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  mark_whole(h, L);
  return NAVGPU_OK;
}

int navgpu_grid_layer_touch(navgpu_costmap* h, int layer, uint32_t x, uint32_t y, uint32_t w, uint32_t hgt) {
  Layer* L = get_layer(h, layer, 0);
  if (!L) return fail(NAVGPU_ERR_INVALID, "bad grid layer");
  L->ux = x; L->uy = y; L->uw = w; L->uh = hgt;
  L->updated = true;
  return NAVGPU_OK;
}

int navgpu_layer_set_enabled(navgpu_costmap* h, int layer, int enabled) {
  Layer* L = get_layer(h, layer, -1);
  if (h) h->content_changed = true;
  if (!L) return fail(NAVGPU_ERR_INVALID, "bad layer");
  if (L->kind == 2 && L->enabled != (enabled != 0)) L->need_reinflation = true;  // reconfigureCB :104-107
  L->enabled = enabled != 0;
  return NAVGPU_OK;
}

// common tail of navgpu_obstacle_set_observations / navgpu_obstacle_set_scans: device buffers for n_floats of xyz,
// the clearing / marking observation tables and the marking scratch; `xyz_host` (nullable) is uploaded
static int install_observations(navgpu_costmap* h, Layer* L, const std::vector<DevObs>& clear, const std::vector<DevObs>& mark,
                                int rays, int marks, const float* xyz_host, size_t n_floats) {
  if (n_floats > L->xyz_capacity) {
    if (L->d_xyz) cudaFree(L->d_xyz);
    L->d_xyz = nullptr;
    NAVGPU_CUDA(cudaMalloc(&L->d_xyz, n_floats * sizeof(float)));
    L->xyz_capacity = n_floats;
  }
  if ((size_t)marks > L->mark_cells_capacity) {
    if (L->d_mark_cells) cudaFree(L->d_mark_cells);
    L->d_mark_cells = nullptr;
    NAVGPU_CUDA(cudaMalloc(&L->d_mark_cells, size_t(marks) * 2 * sizeof(long long)));
    L->mark_cells_capacity = size_t(marks) * 2;
  }
  size_t need = std::max(clear.size(), mark.size());
  if (need > L->obs_capacity) {
    if (L->d_clear) cudaFree(L->d_clear);
    if (L->d_mark) cudaFree(L->d_mark);
    NAVGPU_CUDA(cudaMalloc(&L->d_clear, need * sizeof(DevObs)));
    NAVGPU_CUDA(cudaMalloc(&L->d_mark, need * sizeof(DevObs)));
    L->obs_capacity = need;
  }
  // The uploads go through a pinned staging buffer owned by the layer, so they are asynchronous and the call does not
  // have to wait for the stream: [xyz | clearing table | marking table].  The buffer is reused by the next call once
  // the copies that read it have completed (event).
  // (k_obstacle_update takes tables of up to kInlineObs observations in its kernel parameters: no upload then)
  const bool tables_inline = !L->voxel && clear.size() <= (size_t)kInlineObs && mark.size() <= (size_t)kInlineObs;
  const size_t xyz_bytes = xyz_host ? n_floats * sizeof(float) : 0,
               clear_bytes = tables_inline ? 0 : clear.size() * sizeof(DevObs),
               mark_bytes = tables_inline ? 0 : mark.size() * sizeof(DevObs);
  const size_t stage_bytes = ((xyz_bytes + 15) & ~size_t(15)) + clear_bytes + mark_bytes;
  if (stage_bytes > 0) {
    if (!L->ev_stage) NAVGPU_CUDA(cudaEventCreateWithFlags(&L->ev_stage, cudaEventDisableTiming));
    else NAVGPU_CUDA(cudaEventSynchronize(L->ev_stage));
    if (stage_bytes > L->stage_capacity) {
      if (L->h_stage) cudaFreeHost(L->h_stage);
      L->h_stage = nullptr;
      NAVGPU_CUDA(cudaMallocHost(&L->h_stage, 2 * stage_bytes));
      L->stage_capacity = 2 * stage_bytes;
    }
    char* st = L->h_stage;
    char* st_clear = st + ((xyz_bytes + 15) & ~size_t(15));
    char* st_mark = st_clear + clear_bytes;
    if (xyz_bytes) {
      memcpy(st, xyz_host, xyz_bytes);
      NAVGPU_CUDA(cudaMemcpyAsync(L->d_xyz, st, xyz_bytes, cudaMemcpyHostToDevice, h->stream));
    }
    if (clear_bytes) {
      memcpy(st_clear, clear.data(), clear_bytes);
      NAVGPU_CUDA(cudaMemcpyAsync(L->d_clear, st_clear, clear_bytes, cudaMemcpyHostToDevice, h->stream));
    }
    if (mark_bytes) {
      memcpy(st_mark, mark.data(), mark_bytes);
      NAVGPU_CUDA(cudaMemcpyAsync(L->d_mark, st_mark, mark_bytes, cudaMemcpyHostToDevice, h->stream));
    }
    NAVGPU_CUDA(cudaEventRecord(L->ev_stage, h->stream));
  }
  L->n_clear = (int)clear.size();
  L->n_mark = (int)mark.size();
  L->h_clear = clear;
  L->h_mark = mark;
  L->total_rays = rays;
  L->total_marks = marks;
  return NAVGPU_OK;
}

int navgpu_obstacle_set_observations(navgpu_costmap* h, int layer, const navgpu_observation* obs, int n_obs) {
  Layer* L = get_layer(h, layer, 1);
  if (!L || n_obs < 0 || (n_obs > 0 && !obs)) return fail(NAVGPU_ERR_INVALID, "bad obstacle layer / observations");
  NAVGPU_TRY(use_device(h));
  std::vector<float> xyz;
  std::vector<DevObs> clear, mark;
  L->obs.clear();
  int rays = 0, marks = 0;
  double bx0 = 1e300, by0 = 1e300, bx1 = -1e300, by1 = -1e300;
  bool finite = true;
  for (int i = 0; i < n_obs; ++i) {
    if (obs[i].n_points < 0 || (obs[i].n_points > 0 && !obs[i].xyz)) return fail(NAVGPU_ERR_INVALID, "bad observation %d", i);
    bx0 = std::min(bx0, obs[i].origin_x); bx1 = std::max(bx1, obs[i].origin_x);
    by0 = std::min(by0, obs[i].origin_y); by1 = std::max(by1, obs[i].origin_y);
    finite = finite && std::isfinite(obs[i].origin_x) && std::isfinite(obs[i].origin_y);
    float fx0 = INFINITY, fy0 = INFINITY, fx1 = -INFINITY, fy1 = -INFINITY;
    for (int p = 0; p < obs[i].n_points; ++p) {  // NaN points never win a comparison; the kernels drop them too
      const float x = obs[i].xyz[3 * p], y = obs[i].xyz[3 * p + 1];
      fx0 = x < fx0 ? x : fx0; fx1 = x > fx1 ? x : fx1;
      fy0 = y < fy0 ? y : fy0; fy1 = y > fy1 ? y : fy1;
    }
    if (fx1 >= fx0) { bx0 = std::min(bx0, (double)fx0); bx1 = std::max(bx1, (double)fx1); }
    if (fy1 >= fy0) { by0 = std::min(by0, (double)fy0); by1 = std::max(by1, (double)fy1); }
    DevObs d;
    d.ox = obs[i].origin_x; d.oy = obs[i].origin_y; d.oz = obs[i].origin_z;
    d.obstacle_range = obs[i].obstacle_range;
    d.raytrace_range = obs[i].raytrace_range;
    d.first_point = (int)(xyz.size() / 3);
    d.n_points = obs[i].n_points;
    d.flags = (obs[i].marking ? 1 : 0) | (obs[i].clearing ? 2 : 0);
    L->obs.push_back(HostObs{d.ox, d.oy, d.oz, d.obstacle_range, d.raytrace_range, d.first_point, d.n_points,
                             obs[i].marking != 0, obs[i].clearing != 0});
    xyz.insert(xyz.end(), obs[i].xyz, obs[i].xyz + 3 * size_t(obs[i].n_points));
    if (obs[i].clearing && d.n_points > 0) {
      d.first_ray = rays;
      rays += d.n_points;
      clear.push_back(d);
    }
    if (obs[i].marking && d.n_points > 0) {
      d.first_ray = marks;
      marks += d.n_points;
      mark.push_back(d);
    }
  }
  L->touch_box_valid = finite;
  L->tbx0 = bx0; L->tby0 = by0; L->tbx1 = bx1; L->tby1 = by1;
  return install_observations(h, L, clear, mark, rays, marks, xyz.data(), xyz.size());
}

}  // extern "C"

// One scan's projection record (k_project_scans) and observation (DevObs; first_ray is left to the caller) whose points
// start at `first_point` of the cloud and whose ranges / sensor-frame points start at `first_range` of the upload.
static void scan_record(const navgpu_laser_scan& sc, int first_point, int first_range, ScanRec& r, DevObs& d) {
  r.angle_min = sc.angle_min;
  r.angle_increment = sc.angle_increment;
  r.range_min = sc.range_min;
  r.range_max = sc.range_max;
  sensor_affine(sc.sensor_to_global_rotation_xyzw, sc.sensor_to_global_translation, r.m, r.t);
  r.min_obstacle_height = sc.min_obstacle_height;
  r.max_obstacle_height = sc.max_obstacle_height;
  r.inf_is_valid = sc.inf_is_valid;
  r.first_point = first_point;
  r.n_points = sc.n_ranges;
  r.first_range = first_range;
  r.is_cloud = sc.is_cloud != 0;
  // the sensor origin is the transform of (0, 0, 0): its translation (observation_buffer.cpp:143-151)
  d.ox = sc.sensor_to_global_translation[0]; d.oy = sc.sensor_to_global_translation[1]; d.oz = sc.sensor_to_global_translation[2];
  d.obstacle_range = sc.obstacle_range;
  d.raytrace_range = sc.raytrace_range;
  d.first_point = first_point;
  d.n_points = sc.n_ranges;
  d.first_ray = 0;
  d.flags = (sc.marking ? 1 : 0) | (sc.clearing ? 2 : 0);
}

extern "C" {

// Observation ingest on the device: see k_project_scans (costmap_kernels.cuh) for what is computed and which
// reference / third-party code it stands for.
int navgpu_obstacle_set_scans(navgpu_costmap* h, int layer, const navgpu_laser_scan* scans, int n_scans) {
  Layer* L = get_layer(h, layer, 1);
  if (!L || n_scans < 0 || (n_scans > 0 && !scans)) return fail(NAVGPU_ERR_INVALID, "bad obstacle layer / scans");
  NAVGPU_TRY(use_device(h));
  L->touch_box_valid = false;  // the projected points only ever exist on the device
  std::vector<float> ranges;
  std::vector<ScanRec> recs;
  std::vector<DevObs> clear, mark;
  L->obs.clear();
  int rays = 0, marks = 0, points = 0;
  for (int i = 0; i < n_scans; ++i) {
    const navgpu_laser_scan& sc = scans[i];
    if (sc.n_ranges < 0 || (sc.n_ranges > 0 && !sc.ranges)) return fail(NAVGPU_ERR_INVALID, "bad scan %d", i);
    ScanRec r;
    DevObs d;
    scan_record(sc, points, (int)ranges.size(), r, d);
    ranges.insert(ranges.end(), sc.ranges, sc.ranges + size_t(sc.n_ranges) * (sc.is_cloud ? 3 : 1));
    recs.push_back(r);
    L->obs.push_back(HostObs{d.ox, d.oy, d.oz, d.obstacle_range, d.raytrace_range, d.first_point, d.n_points, sc.marking != 0,
                             sc.clearing != 0});
    if (sc.clearing && d.n_points > 0) { d.first_ray = rays; rays += d.n_points; clear.push_back(d); }
    if (sc.marking && d.n_points > 0) { d.first_ray = marks; marks += d.n_points; mark.push_back(d); }
    points += sc.n_ranges;
  }
  NAVGPU_TRY(install_observations(h, L, clear, mark, rays, marks, nullptr, size_t(points) * 3));
  if (points == 0) return NAVGPU_OK;
  const size_t need = ranges.size() * sizeof(float) + recs.size() * sizeof(ScanRec);
  if (need > L->scan_capacity) {
    if (L->d_scan) cudaFree(L->d_scan);
    L->d_scan = nullptr;
    NAVGPU_CUDA(cudaMalloc(&L->d_scan, 2 * need));
    L->scan_capacity = 2 * need;
  }
  ScanRec* d_recs = reinterpret_cast<ScanRec*>(L->d_scan);  // records first (8-byte aligned), ranges behind them
  float* d_ranges = reinterpret_cast<float*>(L->d_scan + recs.size() * sizeof(ScanRec));
  NAVGPU_CUDA(cudaMemcpyAsync(d_recs, recs.data(), recs.size() * sizeof(ScanRec), cudaMemcpyHostToDevice, h->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(d_ranges, ranges.data(), ranges.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  k_project_scans<<<(points + 255) / 256, 256, 0, h->stream>>>(d_recs, (int)recs.size(), d_ranges, L->d_xyz, points);
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));  // the staging vectors above are pageable
  return NAVGPU_OK;
}

int navgpu_obstacle_get_cloud(navgpu_costmap* h, int layer, int index, float* xyz_out, int capacity, int* n_out) {
  Layer* L = get_layer(h, layer, 1);
  if (!L || !n_out || index < 0 || index >= (int)L->obs.size() || capacity < 0 || (capacity > 0 && !xyz_out))
    return fail(NAVGPU_ERR_INVALID, "bad arguments");
  NAVGPU_TRY(use_device(h));
  const HostObs& o = L->obs[index];
  std::vector<float> tmp(size_t(o.n_points) * 3);
  if (o.n_points > 0) {
    NAVGPU_CUDA(cudaMemcpyAsync(tmp.data(), L->d_xyz + size_t(o.first_point) * 3, tmp.size() * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  }
  int n = 0;
  for (int i = 0; i < o.n_points; ++i) {
    if (tmp[3 * i] != tmp[3 * i]) continue;  // a dropped ray
    if (n < capacity) memcpy(xyz_out + 3 * n, &tmp[3 * i], 3 * sizeof(float));
    ++n;
  }
  *n_out = n;
  return NAVGPU_OK;
}

int navgpu_inflation_set_params(navgpu_costmap* h, int layer, double inflation_radius, double cost_scaling_factor) {
  Layer* L = get_layer(h, layer, 2);
  if (h) h->content_changed = true;
  if (!L) return fail(NAVGPU_ERR_INVALID, "bad inflation layer");
  if (L->weight != cost_scaling_factor || L->radius != inflation_radius) {  // inflation_layer.cpp:356-370
    L->radius = inflation_radius;
    L->weight = cost_scaling_factor;
    L->need_reinflation = true;
    L->tables_dirty = true;
  }
  return NAVGPU_OK;
}

int navgpu_inflation_set_mode(navgpu_costmap* h, int layer, int mode) {
  Layer* L = get_layer(h, layer, 2);
  if (h) h->content_changed = true;
  if (!L || mode < 0 || mode > 1) return fail(NAVGPU_ERR_INVALID, "bad inflation layer / mode");
  if (L->mode != mode) L->tables_dirty = true;  // mode 1 keeps the 2-D rank / cost tables on the device
  L->mode = mode;
  return NAVGPU_OK;
}

int navgpu_inflation_last_rounds(navgpu_costmap* h, int* rounds_out) {
  if (!h || !rounds_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  *rounds_out = 0;
  if (!h->d_prop_ctl) return NAVGPU_OK;
  NAVGPU_TRY(use_device(h));
  unsigned r = 0;
  NAVGPU_CUDA(cudaMemcpyAsync(&r, &h->d_prop_ctl->rounds, sizeof(r), cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  *rounds_out = (int)r;
  return NAVGPU_OK;
}

int navgpu_costmap_force_generic_sweep(navgpu_costmap* h, int enabled) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  h->content_changed = true;
  h->force_generic = enabled != 0;
  return NAVGPU_OK;
}

int navgpu_costmap_set_profiling(navgpu_costmap* h, int enabled) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  NAVGPU_TRY(use_device(h));
  if (enabled && !h->ev_sweep[0]) {
    for (int i = 0; i < 2; ++i) {
      NAVGPU_CUDA(cudaEventCreate(&h->ev_sweep[i]));
      NAVGPU_CUDA(cudaEventCreate(&h->ev_cycle[i]));
    }
    NAVGPU_CUDA(cudaEventCreate(&h->ev_mid));
  }
  h->profile = enabled != 0;
  return NAVGPU_OK;
}

int navgpu_costmap_last_timing(navgpu_costmap* h, float* cycle_ms, float* sweep_ms) {
  if (!h || !h->profile) return fail(NAVGPU_ERR_INVALID, "profiling is not enabled on this handle");
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaEventSynchronize(h->ev_cycle[1]));
  if (cycle_ms) NAVGPU_CUDA(cudaEventElapsedTime(cycle_ms, h->ev_cycle[0], h->ev_cycle[1]));
  if (sweep_ms) NAVGPU_CUDA(cudaEventElapsedTime(sweep_ms, h->ev_sweep[0], h->ev_sweep[1]));
  return NAVGPU_OK;
}

int navgpu_costmap_update_map_async(navgpu_costmap* h, double rx, double ry, double ryaw) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  if (h->profile) cudaEventRecord(h->ev_cycle[0], h->stream);
  NAVGPU_TRY(enqueue_update(h, rx, ry, ryaw));
  if (h->profile) cudaEventRecord(h->ev_cycle[1], h->stream);
  NAVGPU_CUDA(cudaGetLastError());
  return NAVGPU_OK;
}

int navgpu_costmap_synchronize(navgpu_costmap* h) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

int navgpu_costmap_update_map(navgpu_costmap* h, double rx, double ry, double ryaw, int32_t window_out[4]) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  NAVGPU_TRY(enqueue_update(h, rx, ry, ryaw));
  NAVGPU_CUDA(cudaGetLastError());
  if (!h->layers.empty())
    NAVGPU_CUDA(cudaMemcpyAsync(h->h_win, h->d_win, sizeof(DevWindow), cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  if (!h->layers.empty()) {
    h->win[0] = h->h_win->x0; h->win[1] = h->h_win->xn; h->win[2] = h->h_win->y0; h->win[3] = h->h_win->yn;
  }
  if (window_out)
    for (int i = 0; i < 4; ++i) window_out[i] = h->win[i];
  return NAVGPU_OK;
}

int navgpu_costmap_last_timing_split(navgpu_costmap* h, float* merge_ms, float* inflate_ms) {
  if (!h || !h->profile) return fail(NAVGPU_ERR_INVALID, "profiling is not enabled on this handle");
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaEventSynchronize(h->ev_sweep[1]));
  if (merge_ms) NAVGPU_CUDA(cudaEventElapsedTime(merge_ms, h->ev_sweep[0], h->ev_mid));
  if (inflate_ms) NAVGPU_CUDA(cudaEventElapsedTime(inflate_ms, h->ev_mid, h->ev_sweep[1]));
  return NAVGPU_OK;
}

void* navgpu_costmap_stream(navgpu_costmap* h) { return h ? (void*)h->stream : nullptr; }

int navgpu_costmap_get_window(navgpu_costmap* h, int x0, int y0, int xn, int yn, uint8_t* host_out) {
  if (!h || !host_out || x0 < 0 || y0 < 0 || xn > (int)h->sx || yn > (int)h->sy || xn < x0 || yn < y0)
    return fail(NAVGPU_ERR_INVALID, "bad window");
  if (xn == x0 || yn == y0) return NAVGPU_OK;
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaMemcpy2DAsync(host_out, xn - x0, h->master[h->cur] + size_t(y0) * h->pitch + x0, h->pitch, xn - x0,
                                yn - y0, cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

int navgpu_costmap_get_window_into(navgpu_costmap* h, int x0, int y0, int xn, int yn, uint8_t* host_grid, uint32_t host_pitch) {
  if (!h || !host_grid || x0 < 0 || y0 < 0 || xn > (int)h->sx || yn > (int)h->sy || xn < x0 || yn < y0 || host_pitch < h->sx)
    return fail(NAVGPU_ERR_INVALID, "bad window");
  if (xn == x0 || yn == y0) return NAVGPU_OK;
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaMemcpy2DAsync(host_grid + size_t(y0) * host_pitch + x0, host_pitch,
                                h->master[h->cur] + size_t(y0) * h->pitch + x0, h->pitch, xn - x0, yn - y0,
                                cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

// ---- host mirror ---------------------------------------------------------------------------------------------------
int navgpu_costmap_mirror_invalidate(navgpu_costmap* h) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  h->shadow_valid = false;
  return NAVGPU_OK;
}

int navgpu_costmap_get_changed(navgpu_costmap* h, uint8_t* host_grid, uint32_t host_pitch, int32_t* rects_out,
                               int rects_capacity, int32_t* n_rects_out, uint64_t* d2h_bytes_out) {
  if (!h || !host_grid || host_pitch < h->sx || rects_capacity < 0 || (rects_capacity > 0 && !rects_out))
    return fail(NAVGPU_ERR_INVALID, "bad arguments");
  NAVGPU_TRY(use_device(h));
  const unsigned tiles_x = (h->sx + kMirrorTileW - 1) / kMirrorTileW, tiles_y = (h->sy + kMirrorTileH - 1) / kMirrorTileH;
  const unsigned n_tiles = tiles_x * tiles_y;
  if (!h->d_shadow) {
    // staging for up to a quarter of the grid (at least 64 tiles, at most 4 MB): beyond that one plain copy is cheaper
    h->mirror_capacity = std::max(64u, std::min(2048u, n_tiles / 4));
    NAVGPU_CUDA(cudaMalloc(&h->d_shadow, h->bytes()));
    NAVGPU_CUDA(cudaMalloc(&h->d_mirror_counters, 2 * sizeof(unsigned)));
    NAVGPU_CUDA(cudaMemsetAsync(h->d_mirror_counters, 0, 2 * sizeof(unsigned), h->stream));
    NAVGPU_CUDA(cudaHostAlloc(&h->h_mirror_stage, size_t(h->mirror_capacity) * kMirrorTileBytes, cudaHostAllocMapped));
    NAVGPU_CUDA(cudaHostAlloc(&h->h_mirror_tiles, size_t(h->mirror_capacity) * sizeof(unsigned), cudaHostAllocMapped));
    NAVGPU_CUDA(cudaHostAlloc(&h->h_mirror_ctl, sizeof(MirrorCtl), cudaHostAllocMapped));
    memset(h->h_mirror_ctl, 0, sizeof(MirrorCtl));
    h->shadow_valid = false;
  }
  if (host_grid != h->mirror_host || host_pitch != h->mirror_host_pitch) h->shadow_valid = false;
  auto whole_grid = [&]() -> int {
    NAVGPU_CUDA(cudaMemcpy2DAsync(host_grid, host_pitch, h->master[h->cur], h->pitch, h->sx, h->sy, cudaMemcpyDeviceToHost,
                                  h->stream));
    return NAVGPU_OK;
  };
  auto report_whole = [&]() {
    if (n_rects_out) *n_rects_out = 1;
    if (rects_capacity > 0) { rects_out[0] = 0; rects_out[1] = 0; rects_out[2] = (int)h->sx; rects_out[3] = (int)h->sy; }
    if (d2h_bytes_out) *d2h_bytes_out = uint64_t(h->sx) * h->sy;
  };
  if (!h->shadow_valid) {
    NAVGPU_TRY(whole_grid());
    NAVGPU_CUDA(cudaMemcpyAsync(h->d_shadow, h->master[h->cur], h->bytes(), cudaMemcpyDeviceToDevice, h->stream));
    if (!h->layers.empty())
      NAVGPU_CUDA(cudaMemcpyAsync(h->h_win, h->d_win, sizeof(DevWindow), cudaMemcpyDeviceToHost, h->stream));
    NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
    if (!h->layers.empty()) {
      h->win[0] = h->h_win->x0; h->win[1] = h->h_win->xn; h->win[2] = h->h_win->y0; h->win[3] = h->h_win->yn;
    }
    h->shadow_valid = true;
    h->mirror_host = host_grid;
    h->mirror_host_pitch = host_pitch;
    NAVGPU_CUDA(cudaMemsetAsync(h->d_mirror_dirty, 0, sizeof(DevWindow), h->stream));
    h->mirror_all = false;
    h->refine_valid = true;
    h->refine[0] = h->refine[1] = h->refine[2] = h->refine[3] = 0;
    report_whole();
    return NAVGPU_OK;
  }
  MirrorArgs a;
  a.master = h->master[h->cur];
  a.shadow = h->d_shadow;
  a.sx = h->sx; a.sy = h->sy; a.pitch = h->pitch;
  a.tiles_x = tiles_x; a.tiles_y = tiles_y;
  a.capacity = h->mirror_capacity;
  a.stage = h->h_mirror_stage;
  a.stage_tile = h->h_mirror_tiles;
  a.counters = h->d_mirror_counters;
  a.ctl = h->h_mirror_ctl;
  a.win = h->layers.empty() ? nullptr : h->d_win;
  a.dirty = h->d_mirror_dirty;
  a.all = h->mirror_all ? 1 : 0;
  if (h->refine_valid) {
    a.hx0 = h->refine[0]; a.hxn = h->refine[1]; a.hy0 = h->refine[2]; a.hyn = h->refine[3];
  } else {
    a.hx0 = 0; a.hxn = (int)h->sx; a.hy0 = 0; a.hyn = (int)h->sy;
  }
  // a page-locked, mapped mirror (navgpu_host_register, cudaHostAlloc) takes the tiles directly; asked every call, since
  // the caller may have released the registration in between
  a.host_direct = nullptr;
  a.host_pitch = host_pitch;
  {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, host_grid) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer) {
      void* last = nullptr;  // the whole grid must lie inside the registered range: probe its last byte as well
      cudaPointerAttributes attr_end;
      const uint8_t* end_byte = host_grid + size_t(h->sy - 1) * host_pitch + (h->sx - 1);
      if (cudaPointerGetAttributes(&attr_end, end_byte) == cudaSuccess && attr_end.type == cudaMemoryTypeHost && attr_end.devicePointer)
        last = attr_end.devicePointer;
      if (last == static_cast<uint8_t*>(attr.devicePointer) + (end_byte - host_grid)) a.host_direct = static_cast<uint8_t*>(attr.devicePointer);
    } else {
      cudaGetLastError();  // an ordinary pageable pointer is not an error here
    }
  }
  a.tx0 = 0; a.ty0 = 0; a.tw = tiles_x; a.th = tiles_y;
  // (every cycle since the last call was a whole-map cycle on a clean grid: the sweep enqueued last is the only work in
  // flight that writes the cells this call compares)
  const bool mirror_refinable = !a.all && h->refine_valid;
  if (!a.all && h->refine_valid) {  // the host's box bounds the work: launch only the tiles it touches (possibly none)
    a.tx0 = (unsigned)a.hx0 / kMirrorTileW;
    a.ty0 = (unsigned)a.hy0 / kMirrorTileH;
    a.tw = a.hxn > a.hx0 ? ((unsigned)a.hxn + kMirrorTileW - 1) / kMirrorTileW - a.tx0 : 0u;
    a.th = a.hyn > a.hy0 ? ((unsigned)a.hyn + kMirrorTileH - 1) / kMirrorTileH - a.ty0 : 0u;
  }
  h->mirror_all = false;
  h->refine_valid = true;  // from here on: until a cycle that is not of the refinable kind
  h->refine[0] = h->refine[1] = h->refine[2] = h->refine[3] = 0;
  const unsigned launched_tiles = std::max(1u, a.tw * a.th);  // (one CTA at least: it publishes the counts and the window)
  if (mirror_refinable && h->inflate_done_epoch != 0) {
    a.inflate_done = h->d_inflate_done;
    a.inflate_epoch = h->inflate_done_epoch;
    a.inflate_pitch = h->inflate_done_pitch;
  }
  a.seq = ++h->mirror_seq;
  NAVGPU_CUDA(launch_pdl(k_mirror_diff, dim3((launched_tiles + kMirrorWarps - 1) / kMirrorWarps), dim3(kMirrorWarps * 32), 0,
                         h->stream, a));
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaGetLastError());
  {  // wait for the kernel's last word in mapped memory; a stream synchronisation backs the poll up (errors, hangs)
    const volatile unsigned* seq = &h->h_mirror_ctl->seq;
    bool seen = false;
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned spin = 0;; ++spin) {
      if (*seq == a.seq) { seen = true; break; }
      if ((spin & 1023u) == 1023u && std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(2)) break;
#if defined(__x86_64__)
      __builtin_ia32_pause();
#endif
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    if (!seen) NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  }
  const MirrorCtl& ctl = *h->h_mirror_ctl;
  if (a.win) { h->win[0] = ctl.win.x0; h->win[1] = ctl.win.xn; h->win[2] = ctl.win.y0; h->win[3] = ctl.win.yn; }
  if (ctl.n_changed > h->mirror_capacity && !a.host_direct) {  // the shadow is up to date already; the host takes the plain copy
    NAVGPU_TRY(whole_grid());
    NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
    report_whole();
    return NAVGPU_OK;
  }
  if (ctl.n_changed > h->mirror_capacity) {  // direct mode: the data is in place, only the tile list overflowed
    if (n_rects_out) *n_rects_out = std::max((int)ctl.n_changed, rects_capacity + 1);  // "treat the whole grid as changed"
    if (rects_capacity > 0) { rects_out[0] = 0; rects_out[1] = 0; rects_out[2] = (int)h->sx; rects_out[3] = (int)h->sy; }
    if (d2h_bytes_out) *d2h_bytes_out = uint64_t(ctl.n_changed) * kMirrorTileBytes + sizeof(MirrorCtl);
    return NAVGPU_OK;
  }
  const unsigned n = ctl.n_staged;
  for (unsigned k = 0; k < n; ++k) {
    const unsigned t = h->h_mirror_tiles[k], tx = t % tiles_x, ty = t / tiles_x;
    const unsigned x0 = tx * kMirrorTileW, y0 = ty * kMirrorTileH;
    const unsigned w = std::min<unsigned>(kMirrorTileW, h->sx - x0), hg = std::min<unsigned>(kMirrorTileH, h->sy - y0);
    if (!a.host_direct) {
      const uint8_t* src = h->h_mirror_stage + size_t(k) * kMirrorTileBytes;
      uint8_t* dst = host_grid + size_t(y0) * host_pitch + x0;
      for (unsigned r = 0; r < hg; ++r) memcpy(dst + size_t(r) * host_pitch, src + r * kMirrorTileW, w);
    }
    if ((int)k < rects_capacity) {
      rects_out[4 * k] = (int)x0; rects_out[4 * k + 1] = (int)y0;
      rects_out[4 * k + 2] = (int)(x0 + w); rects_out[4 * k + 3] = (int)(y0 + hg);
    }
  }
  if (n_rects_out) *n_rects_out = (int)n;
  if (d2h_bytes_out) *d2h_bytes_out = uint64_t(n) * (kMirrorTileBytes + sizeof(unsigned)) + sizeof(MirrorCtl);
  return NAVGPU_OK;
}

int navgpu_costmap_last_window(navgpu_costmap* h, int32_t window_out[4]) {
  if (!h || !window_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  for (int i = 0; i < 4; ++i) window_out[i] = h->win[i];
  return NAVGPU_OK;
}

int navgpu_host_register(void* ptr, size_t bytes) {
  if (!ptr || bytes == 0) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (navgpu_device_count() <= 0) return fail(NAVGPU_ERR_CUDA, "no CUDA device (libnavgpu has no CPU fallback)");
  NAVGPU_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
  return NAVGPU_OK;
}

int navgpu_host_unregister(void* ptr) {
  if (!ptr) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  NAVGPU_CUDA(cudaHostUnregister(ptr));
  return NAVGPU_OK;
}

int navgpu_costmap_get_window_occupancy(navgpu_costmap* h, int x0, int y0, int xn, int yn, int8_t* host_out) {
  if (!h || !host_out || x0 < 0 || y0 < 0 || xn > (int)h->sx || yn > (int)h->sy || xn < x0 || yn < y0)
    return fail(NAVGPU_ERR_INVALID, "bad window");
  if (xn == x0 || yn == y0) return NAVGPU_OK;
  NAVGPU_TRY(use_device(h));
  const size_t n = size_t(xn - x0) * (yn - y0);
  if (n > h->occupancy_capacity) {
    if (h->d_occupancy) cudaFree(h->d_occupancy);
    h->d_occupancy = nullptr;
    NAVGPU_CUDA(cudaMalloc(&h->d_occupancy, n));
    h->occupancy_capacity = n;
  }
  const int groups = ((xn + 15) >> 4) - (x0 >> 4);  // 16-cell groups of a master row that the window touches
  dim3 block(256), grid((groups + 255) / 256, yn - y0);
  k_translate_window<<<grid, block, 0, h->stream>>>(h->master[h->cur], h->pitch, x0, y0, xn - x0, yn - y0, h->d_occupancy);
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaMemcpyAsync(host_out, h->d_occupancy, n, cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

int navgpu_costmap_get(navgpu_costmap* h, uint8_t* host_out) {
  if (!h) return fail(NAVGPU_ERR_INVALID, "null handle");
  return navgpu_costmap_get_window(h, 0, 0, h->sx, h->sy, host_out);
}

int navgpu_costmap_set(navgpu_costmap* h, const uint8_t* host_in) {
  if (!h || !host_in) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  h->mirror_all = true;  // the master grid is written behind the update cycles' back
  h->master_clean = false;
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaMemcpy2DAsync(h->master[h->cur], h->pitch, host_in, h->sx, h->sx, h->sy, cudaMemcpyHostToDevice, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

int navgpu_layer_get(navgpu_costmap* h, int layer, uint8_t* host_out) {
  Layer* L = get_layer(h, layer, -1);
  if (!L || !host_out || L->kind == 2) return fail(NAVGPU_ERR_INVALID, "layer has no grid");
  NAVGPU_TRY(use_device(h));
  NAVGPU_CUDA(cudaMemcpy2DAsync(host_out, h->sx, L->grid[L->cur], h->pitch, h->sx, h->sy, cudaMemcpyDeviceToHost, h->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(h->stream));
  return NAVGPU_OK;
}

int navgpu_costmap_get_origin(navgpu_costmap* h, double out[2]) {
  if (!h || !out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  out[0] = h->ox;
  out[1] = h->oy;
  return NAVGPU_OK;
}

int navgpu_costmap_device_grid(navgpu_costmap* h, const uint8_t** dev_ptr, uint32_t* pitch) {
  if (!h || !dev_ptr || !pitch) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  *dev_ptr = h->master[h->cur];
  *pitch = h->pitch;
  return NAVGPU_OK;
}

int navgpu_inflation_tables(navgpu_costmap* h, int layer, uint8_t* costs_out, double* dists_out, int capacity,
                            int* radius_out) {
  Layer* L = get_layer(h, layer, 2);
  if (!L || !radius_out) return fail(NAVGPU_ERR_INVALID, "bad inflation layer");
  CostTables t;
  build_tables(t, cell_distance(L->radius, h->res), h->res, L->inscribed, L->weight);
  *radius_out = (int)t.R;
  int n = (int)t.R + 2;
  if (n * n > capacity) return fail(NAVGPU_ERR_CAPACITY, "table needs %d entries", n * n);
  if (costs_out) memcpy(costs_out, t.costs.data(), size_t(n) * n);
  if (dists_out) memcpy(dists_out, t.dists.data(), size_t(n) * n * sizeof(double));
  return NAVGPU_OK;
}

int navgpu_build_cost_table(double resolution, double inscribed_radius, double inflation_radius,
                            double cost_scaling_factor, uint8_t* costs_out, double* dists_out, int capacity,
                            int* radius_out) {
  if (!(resolution > 0) || !radius_out) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  CostTables t;
  build_tables(t, cell_distance(inflation_radius, resolution), resolution, inscribed_radius, cost_scaling_factor);
  *radius_out = (int)t.R;
  int n = (int)t.R + 2;
  if (n * n > capacity) return fail(NAVGPU_ERR_CAPACITY, "table needs %d entries", n * n);
  if (costs_out) memcpy(costs_out, t.costs.data(), size_t(n) * n);
  if (dists_out) memcpy(dists_out, t.dists.data(), size_t(n) * n * sizeof(double));
  return NAVGPU_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------------------------
// Stateless plugin-seam calls on a HOST master grid (include/navgpu.h): the body of a costmap_2d::Layer::updateCosts
// override.  Rows [min_j - 2R, max_j + 2R) are staged to the device (the only rows the reference can read or write,
// inflation_layer.cpp:203-264), processed by the same k_update_costs kernel, and copied back.
namespace {

struct SeamContext {
  int device = -1;
  cudaStream_t stream = nullptr;
  uint8_t* d_master = nullptr;
  uint8_t* d_layer = nullptr;
  uint8_t* d_table = nullptr;
  DevWindow* d_win = nullptr;
  uint16_t* d_seeds = nullptr;
  size_t cap_master = 0, cap_layer = 0, cap_table = 0, cap_seeds = 0;
  unsigned seeds_pitch = 0;
};

int seam_context(int device, SeamContext** out) {
  static thread_local SeamContext ctx[16];
  if (device < 0 || device >= 16) return fail(NAVGPU_ERR_INVALID, "bad device %d", device);
  if (navgpu_device_count() <= device) return fail(NAVGPU_ERR_CUDA, "no CUDA device %d (libnavgpu has no CPU fallback)", device);
  SeamContext& c = ctx[device];
  NAVGPU_CUDA(cudaSetDevice(device));
  if (c.device < 0) {
    NAVGPU_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    NAVGPU_CUDA(cudaMalloc(&c.d_win, sizeof(DevWindow)));
    c.device = device;
  }
  *out = &c;
  return NAVGPU_OK;
}

int ensure(uint8_t** p, size_t* cap, size_t need) {
  if (need <= *cap) return NAVGPU_OK;
  if (*p) cudaFree(*p);
  *p = nullptr;
  NAVGPU_CUDA(cudaMalloc(p, need));
  *cap = need;
  return NAVGPU_OK;
}

int seam_run(uint8_t* master, const uint8_t* layer, uint32_t size_x, uint32_t size_y, int min_i, int min_j, int max_i,
             int max_j, int policy, const uint8_t* by_d2, int R, int device) {
  SeamContext* c;
  NAVGPU_TRY(seam_context(device, &c));
  if (max_i <= min_i || max_j <= min_j) return NAVGPU_OK;
  const int y_lo = std::max(0, min_j - 2 * R), y_hi = std::min((int)size_y, max_j + 2 * R);
  if (y_hi <= y_lo) return NAVGPU_OK;
  const unsigned rows = y_hi - y_lo, pitch = grid_pitch(size_x);
  NAVGPU_TRY(ensure(&c->d_master, &c->cap_master, size_t(pitch) * rows));
  NAVGPU_CUDA(cudaMemcpy2DAsync(c->d_master, pitch, master + size_t(y_lo) * size_x, size_x, size_x, rows,
                                cudaMemcpyHostToDevice, c->stream));
  MergeLayers ml;
  ml.n = 0;
  if (layer) {
    NAVGPU_TRY(ensure(&c->d_layer, &c->cap_layer, size_t(pitch) * rows));
    NAVGPU_CUDA(cudaMemcpy2DAsync(c->d_layer, pitch, layer + size_t(y_lo) * size_x, size_x, size_x, rows,
                                  cudaMemcpyHostToDevice, c->stream));
    ml.n = 1;
    ml.grid[0] = c->d_layer;
    ml.policy[0] = policy;
  }
  if (R > 0) {
    NAVGPU_TRY(ensure(&c->d_table, &c->cap_table, size_t(R) * R + 1 + 8));  // (staged by 32-bit words)
    NAVGPU_CUDA(cudaMemcpyAsync(c->d_table, by_d2, size_t(R) * R + 1, cudaMemcpyHostToDevice, c->stream));
  }
  k_set_window<<<1, 32, 0, c->stream>>>(c->d_win, min_i, max_i, min_j - y_lo, max_j - y_lo);
  UpdateArgs a;
  a.master = c->d_master;
  a.sx = size_x; a.sy = rows; a.pitch = pitch;
  a.def = 0;
  a.do_reset = 0;
  a.win = c->d_win;
  a.ml = ml;
  a.R = R;
  a.cost_d2 = c->d_table;
  a.reach2 = 0;
  for (int d2 = 0; R > 0 && d2 <= R * R; ++d2)
    if (by_d2[d2] != 0) a.reach2 = d2;
  if (R > 0 && R <= 31) {
    NAVGPU_TRY(ensure_seeds(&c->d_seeds, &c->cap_seeds, pitch, rows, c->stream));
    if (c->seeds_pitch != pitch) {  // another row layout: the pad groups of the new layout must read as zero
      NAVGPU_CUDA(cudaMemsetAsync(c->d_seeds, 0, c->cap_seeds, c->stream));
      c->seeds_pitch = pitch;
    }
  }
  NAVGPU_TRY(launch_sweep(a, c->d_seeds, c->stream, false));
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaGetLastError());
  NAVGPU_CUDA(cudaMemcpy2DAsync(master + size_t(y_lo) * size_x, size_x, c->d_master, pitch, size_x, rows,
                                cudaMemcpyDeviceToHost, c->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(c->stream));
  return NAVGPU_OK;
}

}  // namespace

extern "C" {

int navgpu_inflate_host(uint8_t* master, uint32_t size_x, uint32_t size_y, int min_i, int min_j, int max_i, int max_j,
                        const uint8_t* cost_table, uint32_t R, int device) {
  if (!master || !cost_table || size_x == 0 || size_y == 0) return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (R == 0) return NAVGPU_OK;
  if (R > 254) return fail(NAVGPU_ERR_UNSUPPORTED, "cell inflation radius %u > 254", R);
  // cached_costs_[dx][dy] -> cost by squared distance; must be consistent (see build_tables)
  const unsigned n = R + 2;
  std::vector<uint8_t> by_d2(size_t(R) * R + 1, 0);
  std::vector<uint8_t> seen(size_t(R) * R + 1, 0);
  for (unsigned i = 0; i < n; ++i)
    for (unsigned j = 0; j < n; ++j) {
      unsigned d2 = i * i + j * j;
      if (d2 > R * R) continue;
      uint8_t cst = cost_table[i * n + j];
      if (seen[d2] && by_d2[d2] != cst)
        return fail(NAVGPU_ERR_UNSUPPORTED, "cost table is not a function of squared distance at (%u,%u)", i, j);
      seen[d2] = 1;
      by_d2[d2] = cst;
    }
  // the window the reference receives is clamped by LayeredCostmap (:117-124); clamp defensively the same way
  min_i = std::max(0, min_i); min_j = std::max(0, min_j);
  max_i = std::min((int)size_x, max_i); max_j = std::min((int)size_y, max_j);
  return seam_run(master, nullptr, size_x, size_y, min_i, min_j, max_i, max_j, NAVGPU_NOTHING, by_d2.data(), (int)R, device);
}

int navgpu_merge_host(uint8_t* master, const uint8_t* layer, uint32_t size_x, uint32_t size_y, int min_i, int min_j,
                      int max_i, int max_j, int policy, int device) {
  if (!master || !layer || size_x == 0 || size_y == 0 || policy < 0 || policy > NAVGPU_NOTHING)
    return fail(NAVGPU_ERR_INVALID, "bad arguments");
  if (min_i < 0 || min_j < 0 || max_i > (int)size_x || max_j > (int)size_y) return fail(NAVGPU_ERR_INVALID, "window outside the grid");
  return seam_run(master, layer, size_x, size_y, min_i, min_j, max_i, max_j, policy, nullptr, 0, device);
}

}  // extern "C"

// ==================================================================================================================
// Sensing fleet (navgpu_fleet_create_sensing, fleet_costmap.cuh): n rolling local costmaps [ObstacleLayer,
// InflationLayer], or [VoxelLayer, InflationLayer] (navgpu_fleet_create_sensing_voxel), updated by k_fleet_costmap, one
// CTA per robot.  The host keeps per robot what navgpu_costmap keeps for
// one: the origin and the observation tables; the cost table is shared.
// ==================================================================================================================
namespace navgpu {

struct FleetCostmap {
  int device = 0, n = 0;
  unsigned sx = 0, sy = 0, pitch = 0, spitch = 0;
  double res = 0;
  navgpu_fleet_costmap_config cm{};
  std::vector<double> fp;  // footprint (x, y) pairs
  uint8_t def = 0;
  CostTables tables;
  size_t smem = 0;
  cudaStream_t stream = nullptr;
  uint8_t* d_layer = nullptr;   // n x sy x pitch
  uint8_t* d_master = nullptr;  // n x sy x pitch
  bool voxel = false;           // the obstacle layer is a VoxelLayer
  VoxelGeom vg{};
  uint32_t* d_vox = nullptr;    // voxel fleets: n x sy x pitch columns
  uint8_t* d_cost_d2 = nullptr;
  DevBox* d_boxes = nullptr;
  InflationBoundsState* d_infl = nullptr;
  DevWindow* d_win = nullptr;
  FleetCmStep* d_steps = nullptr;
  FleetCmStep* h_steps = nullptr;  // pinned
  std::vector<double> origins;     // n x 2, both grids of a robot share it (what the grids on the device were shifted to)
  std::vector<double> rolled;      // n x 2: the origins of the step being enqueued, committed once its kernel is
  bool reinflate = true;           // InflationLayer::need_reinflation_ until the first step
  // sources (navgpu_fleet_set_scans)
  FleetScanRobot* d_robots = nullptr;
  DevObs* d_obs = nullptr;  // clearing table, then marking table
  size_t obs_capacity = 0;
  int n_clear = 0;
  float* d_xyz = nullptr;
  size_t xyz_capacity = 0;
  long long* d_mark_cells = nullptr;
  size_t mark_capacity = 0;
  char* d_scan = nullptr;  // ScanRec records, then ranges
  size_t scan_capacity = 0;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // projection start / end, costmap start / end
  bool projected = false, stepped = false;

  FleetCostmap() = default;
  FleetCostmap(const FleetCostmap&) = delete;
  FleetCostmap& operator=(const FleetCostmap&) = delete;
  ~FleetCostmap() {  // (also what a failed fleet_costmap_create leaves behind)
    cudaSetDevice(device);
    if (stream) cudaStreamSynchronize(stream);
    cudaFree(d_layer); cudaFree(d_master); cudaFree(d_vox); cudaFree(d_cost_d2); cudaFree(d_boxes); cudaFree(d_infl); cudaFree(d_win);
    cudaFree(d_steps); cudaFree(d_robots); cudaFree(d_obs); cudaFree(d_xyz); cudaFree(d_mark_cells); cudaFree(d_scan);
    if (h_steps) cudaFreeHost(h_steps);
    for (cudaEvent_t e : ev)
      if (e) cudaEventDestroy(e);
    if (stream) cudaStreamDestroy(stream);
  }
};

template <typename T>
static int ensure_device(T** p, size_t* cap, size_t n) {
  if (n <= *cap && *p) return NAVGPU_OK;
  if (*p) cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  NAVGPU_CUDA(cudaMalloc(p, std::max<size_t>(1, 2 * n) * sizeof(T)));
  *cap = std::max<size_t>(1, 2 * n);
  return NAVGPU_OK;
}

int fleet_costmap_create(FleetCostmap** out, int n, unsigned sx, unsigned sy, double resolution,
                         const navgpu_fleet_costmap_config& cm, const navgpu_fleet_voxel_config* voxel,
                         const double* footprint_xy, int n_footprint, int device) {
  if (cm.combination_method != 0 && cm.combination_method != 1)
    return fail(NAVGPU_ERR_INVALID, "combination_method %d: 0 (Overwrite) or 1 (Max)", cm.combination_method);
  if (voxel) {  // navgpu_costmap_add_voxel_layer's checks
    const navgpu_fleet_voxel_config& v = *voxel;
    if (v.z_voxels < 0 || v.z_voxels > 16 || !(v.z_resolution > 0) || v.unknown_threshold < 0 || v.mark_threshold < 0)
      return fail(NAVGPU_ERR_INVALID, "bad voxel layer arguments");
    if (v.mark_threshold != 0)
      return fail(NAVGPU_ERR_UNSUPPORTED, "mark_threshold %d: only the reference's default 0 is implemented", v.mark_threshold);
  }
  if (n_footprint > kFleetFootprint) return fail(NAVGPU_ERR_INVALID, "more than %d footprint vertices", kFleetFootprint);
  std::unique_ptr<FleetCostmap> fc(new FleetCostmap);
  FleetCostmap& F = *fc;
  F.device = device;
  F.n = n;
  F.sx = sx; F.sy = sy; F.pitch = grid_pitch(sx); F.spitch = (sx + 3) & ~3u;
  F.res = resolution;
  F.cm = cm;
  F.fp.assign(footprint_xy, footprint_xy + 2 * n_footprint);
  F.def = cm.track_unknown ? kNoInfo : kFree;  // layered_costmap.cpp:53-56, costmap_layer.cpp:14-19
  F.voxel = voxel != nullptr;
  if (voxel)  // VoxelLayer::reconfigureCB (voxel_layer.cpp:84-95): unknown_threshold_ = unknown_threshold + (16 - z_voxels)
    F.vg = VoxelGeom{voxel->origin_z, voxel->z_resolution, (unsigned)voxel->z_voxels,
                     (unsigned)(voxel->unknown_threshold + (16 - voxel->z_voxels)), (unsigned)voxel->mark_threshold};
  std::vector<Pt> fp;
  for (int i = 0; i < n_footprint; ++i) fp.push_back(Pt{footprint_xy[2 * i], footprint_xy[2 * i + 1]});
  double inscribed = 0, circumscribed = 0;
  footprint_radii(fp, inscribed, circumscribed);
  // InflationLayer::computeCaches with the checks of upload_tables
  const unsigned R = cell_distance(cm.inflation_radius, resolution);
  if (R > 254) return fail(NAVGPU_ERR_UNSUPPORTED, "cell inflation radius %u > 254", R);
  build_tables(F.tables, R, resolution, inscribed, cm.cost_scaling_factor);
  if (F.tables.ambiguous)
    return fail(NAVGPU_ERR_UNSUPPORTED, "inflation cost table is not a function of squared distance for R=%u", R);
  // one robot's grids and scratch must fit one CTA's shared memory
  NAVGPU_CUDA(cudaSetDevice(device));
  int smem_optin = 0;
  NAVGPU_CUDA(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  cudaFuncAttributes fa;
  NAVGPU_CUDA(cudaFuncGetAttributes(&fa, F.voxel ? k_fleet_costmap_voxel : k_fleet_costmap));
  F.smem = fleet_costmap_smem(sy, F.spitch, fleet_seed_words(sx), (int)R, F.voxel);
  if (F.smem + fa.sharedSizeBytes > (size_t)smem_optin)
    return fail(NAVGPU_ERR_UNSUPPORTED,
                "a %u x %u map with a cell inflation radius of %u needs %zu B of shared memory per robot; the device allows %d",
                sx, sy, R, F.smem + fa.sharedSizeBytes, smem_optin);
  // the footprint polygon's cells (outline + bounding box, as footprint_polygon counts them) at any pose must fit the
  // rasteriser's scratch: its vertices span at most 2 * circumscribed radius, an edge at most its length + 2 cells
  if (cm.footprint_clearing && n_footprint >= 3) {
    double rc = 0, outline = 0;
    for (int i = 0; i < n_footprint; ++i) {
      const Pt& p = fp[i];
      const Pt& q = fp[(i + 1) % n_footprint];
      rc = std::max(rc, hypot(p.x, p.y));
      outline += std::ceil(hypot(q.x - p.x, q.y - p.y) / resolution) + 2;
    }
    const double span = std::ceil(2 * rc / resolution) + 3;
    if (span * span + outline > kFleetPolyCells)
      return fail(NAVGPU_ERR_UNSUPPORTED, "the footprint polygon can cover %.0f cells; the per-robot rasteriser holds %d",
                  span * span + outline, kFleetPolyCells);
  }
  NAVGPU_CUDA(cudaStreamCreateWithFlags(&F.stream, cudaStreamNonBlocking));
  for (cudaEvent_t& e : F.ev) NAVGPU_CUDA(cudaEventCreate(&e));
  const size_t grid_bytes = size_t(n) * sy * F.pitch;
  NAVGPU_CUDA(cudaMalloc(&F.d_layer, grid_bytes));
  NAVGPU_CUDA(cudaMalloc(&F.d_master, grid_bytes));
  NAVGPU_CUDA(cudaMemset(F.d_layer, F.def, grid_bytes));
  NAVGPU_CUDA(cudaMemset(F.d_master, F.def, grid_bytes));
  if (F.voxel) {  // VoxelGrid starts with all-unknown columns (voxel_grid.cpp:41-59)
    NAVGPU_CUDA(cudaMalloc(&F.d_vox, grid_bytes * sizeof(uint32_t)));
    std::vector<uint32_t> unknown(size_t(sy) * F.pitch, 0x0000ffffu);
    for (int r = 0; r < n; ++r)
      NAVGPU_CUDA(cudaMemcpy(F.d_vox + size_t(r) * sy * F.pitch, unknown.data(), unknown.size() * sizeof(uint32_t),
                             cudaMemcpyHostToDevice));
  }
  NAVGPU_CUDA(cudaMalloc(&F.d_cost_d2, F.tables.by_d2.size()));
  NAVGPU_CUDA(cudaMemcpy(F.d_cost_d2, F.tables.by_d2.data(), F.tables.by_d2.size(), cudaMemcpyHostToDevice));
  NAVGPU_CUDA(cudaMalloc(&F.d_boxes, sizeof(DevBox) * 2 * n));
  NAVGPU_CUDA(cudaMalloc(&F.d_infl, sizeof(InflationBoundsState) * 2 * n));
  NAVGPU_CUDA(cudaMalloc(&F.d_win, sizeof(DevWindow) * n));
  NAVGPU_CUDA(cudaMemset(F.d_win, 0, sizeof(DevWindow) * n));
  {
    const double fm = std::numeric_limits<float>::max();  // inflation_layer.cpp:63-66
    std::vector<DevBox> boxes(size_t(2) * n, DevBox{~0ull, ~0ull, 0ull, 0ull});
    std::vector<InflationBoundsState> infl(size_t(2) * n, InflationBoundsState{-fm, -fm, fm, fm});
    NAVGPU_CUDA(cudaMemcpy(F.d_boxes, boxes.data(), boxes.size() * sizeof(DevBox), cudaMemcpyHostToDevice));
    NAVGPU_CUDA(cudaMemcpy(F.d_infl, infl.data(), infl.size() * sizeof(InflationBoundsState), cudaMemcpyHostToDevice));
  }
  NAVGPU_CUDA(cudaMalloc(&F.d_steps, sizeof(FleetCmStep) * n));
  NAVGPU_CUDA(cudaMallocHost(&F.h_steps, sizeof(FleetCmStep) * n));
  NAVGPU_CUDA(cudaMalloc(&F.d_robots, sizeof(FleetScanRobot) * n));
  NAVGPU_CUDA(cudaMemset(F.d_robots, 0, sizeof(FleetScanRobot) * n));  // no sources yet
  F.origins.assign(size_t(2) * n, 0.0);
  F.rolled = F.origins;
  *out = fc.release();
  return NAVGPU_OK;
}

void fleet_costmap_destroy(FleetCostmap* fc) { delete fc; }

cudaStream_t fleet_costmap_stream(const FleetCostmap* fc) { return fc->stream; }

const uint8_t* fleet_costmap_master(const FleetCostmap* fc, unsigned* pitch) {
  *pitch = fc->pitch;
  return fc->d_master;
}

int fleet_costmap_set_scans(FleetCostmap* fc, const navgpu_laser_scan* scans, const int32_t* offsets) {
  if (!offsets || offsets[0] < 0) return fail(NAVGPU_ERR_INVALID, "bad scan offsets");
  for (int r = 0; r < fc->n; ++r)
    if (offsets[r + 1] < offsets[r]) return fail(NAVGPU_ERR_INVALID, "scan offsets decrease at robot %d", r);
  if (offsets[fc->n] > offsets[0] && !scans) return fail(NAVGPU_ERR_INVALID, "null scans");
  NAVGPU_CUDA(cudaSetDevice(fc->device));
  std::vector<float> ranges;
  std::vector<ScanRec> recs;
  std::vector<DevObs> clear, mark;
  std::vector<FleetScanRobot> robots(fc->n);
  long long points = 0, marks_total = 0;
  for (int r = 0; r < fc->n; ++r) {
    FleetScanRobot& rb = robots[r];
    rb.clear_first = (int)clear.size();
    rb.mark_first = (int)mark.size();
    rb.rays = rb.marks = 0;
    rb.mark_base = marks_total;
    for (int i = offsets[r]; i < offsets[r + 1]; ++i) {
      const navgpu_laser_scan& sc = scans[i];
      if (sc.n_ranges < 0 || (sc.n_ranges > 0 && !sc.ranges)) return fail(NAVGPU_ERR_INVALID, "bad scan %d", i);
      if (points + sc.n_ranges > 0x7fffffffll) return fail(NAVGPU_ERR_UNSUPPORTED, "more than 2^31 scan points");
      ScanRec rec;
      DevObs d;
      scan_record(sc, (int)points, (int)ranges.size(), rec, d);
      ranges.insert(ranges.end(), sc.ranges, sc.ranges + size_t(sc.n_ranges) * (sc.is_cloud ? 3 : 1));
      recs.push_back(rec);
      // a clearing source is listed even without points: raytraceFreespace still touches its origin (:504-521)
      if (sc.clearing) { d.first_ray = rb.rays; rb.rays += sc.n_ranges; clear.push_back(d); }
      if (sc.marking && sc.n_ranges > 0) { d.first_ray = rb.marks; rb.marks += sc.n_ranges; mark.push_back(d); }
      points += sc.n_ranges;
    }
    rb.n_clear = (int)clear.size() - rb.clear_first;
    rb.n_mark = (int)mark.size() - rb.mark_first;
    marks_total += rb.marks;
  }
  for (FleetScanRobot& rb : robots) rb.mark_first += (int)clear.size();  // one table: clearing entries, then marking
  fc->n_clear = (int)clear.size();
  std::vector<DevObs> obs(clear);
  obs.insert(obs.end(), mark.begin(), mark.end());
  NAVGPU_TRY(ensure_device(&fc->d_obs, &fc->obs_capacity, obs.size()));
  NAVGPU_TRY(ensure_device(&fc->d_xyz, &fc->xyz_capacity, size_t(points) * 3));
  NAVGPU_TRY(ensure_device(&fc->d_mark_cells, &fc->mark_capacity, size_t(marks_total)));
  const size_t rec_bytes = recs.size() * sizeof(ScanRec), scan_bytes = rec_bytes + ranges.size() * sizeof(float);
  NAVGPU_TRY(ensure_device(&fc->d_scan, &fc->scan_capacity, scan_bytes));
  if (!obs.empty())
    NAVGPU_CUDA(cudaMemcpyAsync(fc->d_obs, obs.data(), obs.size() * sizeof(DevObs), cudaMemcpyHostToDevice, fc->stream));
  NAVGPU_CUDA(cudaMemcpyAsync(fc->d_robots, robots.data(), robots.size() * sizeof(FleetScanRobot), cudaMemcpyHostToDevice,
                              fc->stream));
  fc->projected = points > 0;
  if (points > 0) {  // every robot's scans in one launch (records first, 8-byte aligned; ranges behind them)
    ScanRec* d_recs = reinterpret_cast<ScanRec*>(fc->d_scan);
    float* d_ranges = reinterpret_cast<float*>(fc->d_scan + rec_bytes);
    NAVGPU_CUDA(cudaMemcpyAsync(d_recs, recs.data(), rec_bytes, cudaMemcpyHostToDevice, fc->stream));
    NAVGPU_CUDA(cudaMemcpyAsync(d_ranges, ranges.data(), ranges.size() * sizeof(float), cudaMemcpyHostToDevice, fc->stream));
    NAVGPU_CUDA(cudaEventRecord(fc->ev[0], fc->stream));
    k_project_scans<<<(unsigned)((points + 255) / 256), 256, 0, fc->stream>>>(d_recs, (int)recs.size(), d_ranges, fc->d_xyz,
                                                                             (int)points);
    NAVGPU_LAUNCHED(1);
    NAVGPU_CUDA(cudaEventRecord(fc->ev[1], fc->stream));
    NAVGPU_CUDA(cudaGetLastError());
  }
  NAVGPU_CUDA(cudaStreamSynchronize(fc->stream));  // the staging vectors above are pageable
  return NAVGPU_OK;
}

bool on_device(const void* p, int device) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();  // not a CUDA pointer at all: clear the error, it is the caller's
    return false;
  }
  return (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) && at.device == device;
}

int fleet_costmap_set_scan_batch(FleetCostmap* fc, const navgpu_fleet_scan_source* sources, int n_sources, bool device) {
  // every check before anything changes: a refused call leaves the previous sources in place
  if (n_sources < 0 || !sources) return fail(NAVGPU_ERR_INVALID, "bad sources");
  if (n_sources > kScanBatchSources)
    return fail(NAVGPU_ERR_UNSUPPORTED, "%d sources: a batch holds up to %d", n_sources, kScanBatchSources);
  const auto bit = [](int32_t v) { return v == 0 || v == 1; };
  long long per_robot = 0;
  for (int s = 0; s < n_sources; ++s) {
    const navgpu_fleet_scan_source& c = sources[s];
    if (!c.sensor_to_global || c.n_points < 0 || (c.n_points > 0 && !c.data) || !bit(c.is_cloud) || !bit(c.marking) ||
        !bit(c.clearing))
      return fail(NAVGPU_ERR_INVALID, "bad source %d", s);
    per_robot += c.n_points;
  }
  if (per_robot * fc->n > 0x7fffffffll) return fail(NAVGPU_ERR_UNSUPPORTED, "more than 2^31 scan points");
  if (device)
    for (int s = 0; s < n_sources; ++s)
      if (!on_device(sources[s].sensor_to_global, fc->device) || (sources[s].n_points > 0 && !on_device(sources[s].data, fc->device)))
        return fail(NAVGPU_ERR_INVALID, "source %d: not device memory of device %d", s, fc->device);
  NAVGPU_CUDA(cudaSetDevice(fc->device));

  // the regular layout of k_fleet_scan_batch, and set_scans' listing rules: a clearing source is listed even without
  // points (raytraceFreespace still touches its origin), a marking source only with points
  ScanBatchArgs a;
  a.n_sources = n_sources;
  a.n = fc->n;
  a.points = a.n_clear = a.n_mark = a.rays = a.marks = 0;
  size_t stage_bytes = 0;  // host variant: every array behind the previous one (transforms 8-byte aligned, first)
  for (int s = 0; s < n_sources; ++s) {
    const navgpu_fleet_scan_source& c = sources[s];
    ScanBatchSource& b = a.src[s];
    b.data = c.data;
    b.stg = c.sensor_to_global;
    b.angle_min = c.angle_min;
    b.angle_increment = c.angle_increment;
    b.min_obstacle_height = c.min_obstacle_height;
    b.max_obstacle_height = c.max_obstacle_height;
    b.obstacle_range = c.obstacle_range;
    b.raytrace_range = c.raytrace_range;
    b.range_min = c.range_min;
    b.range_max = c.range_max;
    b.n_points = c.n_points;
    b.is_cloud = c.is_cloud;
    b.inf_is_valid = c.inf_is_valid;
    b.flags = (c.marking ? 1 : 0) | (c.clearing ? 2 : 0);
    b.point_first = a.points;
    b.clear_slot = b.mark_slot = -1;
    b.clear_ray = b.mark_ray = 0;
    if (c.clearing) { b.clear_slot = a.n_clear++; b.clear_ray = a.rays; a.rays += c.n_points; }
    if (c.marking && c.n_points > 0) { b.mark_slot = a.n_mark++; b.mark_ray = a.marks; a.marks += c.n_points; }
    a.points += c.n_points;
    stage_bytes += size_t(fc->n) * (7 * sizeof(double) + size_t(c.n_points) * (c.is_cloud ? 3 : 1) * sizeof(float));
  }
  const size_t n = size_t(fc->n);
  NAVGPU_TRY(ensure_device(&fc->d_obs, &fc->obs_capacity, n * (a.n_clear + a.n_mark)));
  NAVGPU_TRY(ensure_device(&fc->d_xyz, &fc->xyz_capacity, n * a.points * 3));
  NAVGPU_TRY(ensure_device(&fc->d_mark_cells, &fc->mark_capacity, n * a.marks));
  if (!device) {  // one plain copy per array into the staging buffer, then the device path on the copies
    NAVGPU_TRY(ensure_device(&fc->d_scan, &fc->scan_capacity, stage_bytes));
    char* p = fc->d_scan;
    for (int s = 0; s < n_sources; ++s) {
      const size_t bytes = n * 7 * sizeof(double);
      NAVGPU_CUDA(cudaMemcpyAsync(p, sources[s].sensor_to_global, bytes, cudaMemcpyHostToDevice, fc->stream));
      a.src[s].stg = reinterpret_cast<const double*>(p);
      p += bytes;
    }
    for (int s = 0; s < n_sources; ++s) {
      const size_t bytes = n * sources[s].n_points * (sources[s].is_cloud ? 3 : 1) * sizeof(float);
      if (bytes) NAVGPU_CUDA(cudaMemcpyAsync(p, sources[s].data, bytes, cudaMemcpyHostToDevice, fc->stream));
      a.src[s].data = reinterpret_cast<const float*>(p);
      p += bytes;
    }
  }
  a.xyz = fc->d_xyz;
  a.obs = fc->d_obs;
  a.robots = fc->d_robots;
  long long threads = fc->n;
  for (int s = 0; s < n_sources; ++s) threads = std::max(threads, (long long)fc->n * sources[s].n_points);
  const dim3 grid((unsigned)((threads + kScanBatchThreads - 1) / kScanBatchThreads), (unsigned)std::max(1, n_sources));
  NAVGPU_CUDA(cudaEventRecord(fc->ev[0], fc->stream));
  k_fleet_scan_batch<<<grid, kScanBatchThreads, 0, fc->stream>>>(a);
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaGetLastError());
  NAVGPU_CUDA(cudaEventRecord(fc->ev[1], fc->stream));
  fc->n_clear = fc->n * a.n_clear;
  fc->projected = a.points > 0;
  if (!device) NAVGPU_CUDA(cudaStreamSynchronize(fc->stream));  // the host arrays may be pageable
  return NAVGPU_OK;
}

int fleet_costmap_roll(FleetCostmap* fc, const double* poses, double* origins_xy) {
  // nothing is committed here: a step that fails before its kernel is enqueued leaves the fleet as it was
  for (int r = 0; r < fc->n; ++r) {
    const FleetCmStep st = fleet_roll_step(poses + 3 * r, fc->origins[2 * r], fc->origins[2 * r + 1], fc->sx, fc->sy, fc->res);
    fc->rolled[2 * r] = st.ox;
    fc->rolled[2 * r + 1] = st.oy;
    fc->h_steps[r] = st;
    origins_xy[2 * r] = st.ox;
    origins_xy[2 * r + 1] = st.oy;
  }
  return NAVGPU_OK;
}

FleetCmStep* fleet_costmap_device_steps(FleetCostmap* fc) { return fc->d_steps; }

void fleet_costmap_set_origins(FleetCostmap* fc, const double* origins_xy) {
  fc->origins.assign(origins_xy, origins_xy + size_t(2) * fc->n);
  fc->rolled = fc->origins;
}

int fleet_costmap_enqueue(FleetCostmap* fc, bool device_steps) {
  NAVGPU_CUDA(cudaSetDevice(fc->device));
  if (!device_steps)
    NAVGPU_CUDA(cudaMemcpyAsync(fc->d_steps, fc->h_steps, sizeof(FleetCmStep) * fc->n, cudaMemcpyHostToDevice, fc->stream));
  FleetCostmapArgs a;
  a.layer = fc->d_layer;
  a.vox = fc->d_vox;
  a.v = fc->vg;
  a.master = fc->d_master;
  a.sx = fc->sx; a.sy = fc->sy; a.pitch = fc->pitch; a.spitch = fc->spitch;
  a.res = fc->res;
  a.def = fc->def;
  a.policy = fc->cm.combination_method == 0 ? NAVGPU_OVERWRITE : NAVGPU_MAX;
  a.footprint_clearing = fc->cm.footprint_clearing != 0;
  a.max_obstacle_height = fc->cm.max_obstacle_height;
  a.nfp = (int)(fc->fp.size() / 2);
  for (int k = 0; k < kFleetFootprint; ++k) {
    a.fpx[k] = k < a.nfp ? fc->fp[2 * k] : 0.0;
    a.fpy[k] = k < a.nfp ? fc->fp[2 * k + 1] : 0.0;
  }
  a.robots = fc->d_robots;
  a.steps = fc->d_steps;
  a.clear = fc->d_obs;
  a.mark = fc->d_obs;  // FleetScanRobot::mark_first already counts the clearing entries in front
  a.xyz = fc->d_xyz;
  a.mark_cells = fc->d_mark_cells;
  a.boxes = fc->d_boxes;
  a.infl = fc->d_infl;
  a.win = fc->d_win;
  a.reinflate = fc->reinflate ? 1 : 0;
  a.inflation_radius = fc->cm.inflation_radius;
  a.R = (int)fc->tables.R;
  a.cost_d2 = fc->d_cost_d2;
  // the limit belongs to the kernel, not to this fleet: another fleet (other map size, other radius) may have set its own
  auto* kernel = fc->voxel ? k_fleet_costmap_voxel : k_fleet_costmap;
  NAVGPU_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fc->smem));
  NAVGPU_CUDA(cudaEventRecord(fc->ev[2], fc->stream));
  kernel<<<fc->n, kFleetCmThreads, fc->smem, fc->stream>>>(a);
  NAVGPU_LAUNCHED(1);
  NAVGPU_CUDA(cudaGetLastError());
  NAVGPU_CUDA(cudaEventRecord(fc->ev[3], fc->stream));
  if (!device_steps) fc->origins = fc->rolled;  // the grids on the device now follow the rolled origins
  fc->reinflate = false;
  fc->stepped = true;
  return NAVGPU_OK;
}

int fleet_costmap_get(FleetCostmap* fc, int robot, bool master, uint8_t* host_out) {
  NAVGPU_CUDA(cudaSetDevice(fc->device));
  const uint8_t* src = (master ? fc->d_master : fc->d_layer) + size_t(robot) * fc->sy * fc->pitch;
  NAVGPU_CUDA(cudaMemcpy2DAsync(host_out, fc->sx, src, fc->pitch, fc->sx, fc->sy, cudaMemcpyDeviceToHost, fc->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(fc->stream));
  return NAVGPU_OK;
}

int fleet_costmap_get_voxels(FleetCostmap* fc, int robot, uint32_t* host_out) {
  if (!fc->voxel) return fail(NAVGPU_ERR_INVALID, "not a voxel fleet (navgpu_fleet_create_sensing_voxel)");
  NAVGPU_CUDA(cudaSetDevice(fc->device));
  const uint32_t* src = fc->d_vox + size_t(robot) * fc->sy * fc->pitch;
  NAVGPU_CUDA(cudaMemcpy2DAsync(host_out, fc->sx * sizeof(uint32_t), src, fc->pitch * sizeof(uint32_t),
                                fc->sx * sizeof(uint32_t), fc->sy, cudaMemcpyDeviceToHost, fc->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(fc->stream));
  return NAVGPU_OK;
}

int fleet_costmap_geometry(FleetCostmap* fc, int robot, double origin_out[2], int32_t window_out[4]) {
  NAVGPU_CUDA(cudaSetDevice(fc->device));
  DevWindow w;
  NAVGPU_CUDA(cudaMemcpyAsync(&w, fc->d_win + robot, sizeof(DevWindow), cudaMemcpyDeviceToHost, fc->stream));
  NAVGPU_CUDA(cudaStreamSynchronize(fc->stream));
  origin_out[0] = fc->origins[2 * robot];
  origin_out[1] = fc->origins[2 * robot + 1];
  window_out[0] = w.x0; window_out[1] = w.xn; window_out[2] = w.y0; window_out[3] = w.yn;
  return NAVGPU_OK;
}

int fleet_costmap_last_timing(FleetCostmap* fc, float* project_ms, float* costmap_ms) {
  NAVGPU_CUDA(cudaSetDevice(fc->device));
  NAVGPU_CUDA(cudaStreamSynchronize(fc->stream));
  if (project_ms) {
    *project_ms = 0.0f;
    if (fc->projected) NAVGPU_CUDA(cudaEventElapsedTime(project_ms, fc->ev[0], fc->ev[1]));
  }
  if (costmap_ms) {
    *costmap_ms = 0.0f;
    if (fc->stepped) NAVGPU_CUDA(cudaEventElapsedTime(costmap_ms, fc->ev[2], fc->ev[3]));
  }
  return NAVGPU_OK;
}

}  // namespace navgpu
