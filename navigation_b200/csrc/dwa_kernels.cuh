// dwa_kernels.cuh -- Path B device code: DWA rollout scoring on the GPU (sm_100a).
//
// Reference semantics (file:line under /root/reference) are cited next to each piece; the host side that
// sequences the kernels per DWAPlanner::findBestPath is in dwa.cu.
#pragma once

#include <cstddef>

#include "common.cuh"
#include "fleet_costmap.cuh"

namespace navgpu {

constexpr int kMaxFootprint = 16;
constexpr int kInlineSamples = 640;  // per-axis velocity samples carried in the kernel parameters
constexpr int kDwaWarpsPerBlock = 8;

struct DwaGeom {
  const uint8_t* cost;  // local costmap, row pitch `pitch`
  unsigned sx, sy, pitch;
  double res, ox, oy;
  double inv_res;  // 1 / res, only ever used through exact_cell
};

// (int)(d / res) exactly as IEEE division + truncation gives it, without the fp64 division.
// Fast path: q = d * (1/res) is within a few ulp of d / res, so truncation agrees unless the quotient is within 1e-6
// of an integer r.  Near an integer the decision is made exactly: e = fma(-r, res, d) is the exact value
// of d - r * res (it has at most ~38 significant bits there), so the real quotient is r + e / res.  e >= 0 gives r.
// For e < 0 the correctly rounded quotient still reaches r when r - d/res is at most half the spacing of the doubles
// just below r (a tie rounds to r, whose mantissa is even), i.e. -e <= 2^(k-53) * res with k = floor(log2 r), one less
// when r is a power of two; otherwise the result is r - 1.  (Poses laid out on the grid -- x = 1.5 at 0.05 m cells --
// sit exactly on such borders, so this path is common, not exotic.)
__device__ __forceinline__ int exact_cell(double d, double res, double inv_res) {
  const double q = d * inv_res;
  const double r = rint(q);
  // q is within a few ulp of d / res (|error| < 2e-11 for the map sizes create() accepts, q < 32768), so a fixed
  // 1e-6 band around the integers catches every case in which truncating q could disagree with truncating d / res
  if (fabs(q - r) <= 1e-6) {
    const int ri = (int)r;
    if (ri <= 0) return (int)(d / res);  // d within 1e-9 cells of the origin: keep the division
    const double e = fma(-r, res, d);
    if (e >= 0.0) return ri;
    const int k = 31 - __clz(ri) - (((ri & (ri - 1)) == 0) ? 1 : 0);
    const double half_spacing = __longlong_as_double((long long)(1023 + k - 53) << 52);  // 2^(k - 53)
    return (-e <= half_spacing * res) ? ri : ri - 1;
  }
  return (int)q;
}

__device__ __forceinline__ bool dwa_world_to_map(const DwaGeom& g, double wx, double wy, int& mx, int& my) {
  // Costmap2D::worldToMap, costmap_2d/src/costmap_2d.cpp:208-220
  if (wx < g.ox || wy < g.oy) return false;
  const unsigned ux = (unsigned)exact_cell(wx - g.ox, g.res, g.inv_res), uy = (unsigned)exact_cell(wy - g.oy, g.res, g.inv_res);
  mx = (int)ux;
  my = (int)uy;
  return ux < g.sx && uy < g.sy;
}

// ---------------------------------------------------------------------------------------------------------------
// MapGridCostFunction::prepare for the four grids of DWAPlanner (path, goal, goal_front, alignment):
// MapGrid::resetPathDist + setTargetCells | setLocalGoal + computeTargetDistance
// (base_local_planner/src/map_grid_cost_function.cpp:59-68, src/map_grid.cpp:127-133, 174-310).
//
// One CTA per grid.  The FIFO wavefront with unit edge costs is order independent, so it is evaluated level by level
// on bit planes held in shared memory: frontier F, visited V, passable P, one 32-cell word per thread step:
//     touched = (F<<1 | F>>1 | F(up) | F(down)) & ~V       cells first touched at this level (updatePathCell)
//     dist[touched & ~P] = size_x*size_y (obstacleCosts, not expanded),  dist[touched & P] = level + 1
// A seed is expanded even when it lies on an obstacle, exactly like the reference's queue.  Untouched cells keep
// size_x*size_y + 1 (unreachableCellCosts).
struct MapGridJob {
  const double* plan_xy;  // already passed through MapGrid::adjustPlanResolution on the host (pure plan geometry)
  int n_points;
  int local_goal;  // setLocalGoal (last seed only) vs setTargetCells
  uint32_t* dist;  // sx*sy, row-major, no pitch
  // MapCell::within_robot as a bit per cell ((sx+31)/32 words per row), or null: obstacle cells under it stay
  // passable (map_grid.cpp:109-112; only the legacy TrajectoryPlanner marks cells, trajectory_planner.cpp:918-930)
  const uint32_t* within_robot = nullptr;
  // 1: this grid is identical to another job's (same plan, same mode) whose buffer `dist` already points to -- nothing
  // to compute (DWAPlanner's alignment critic gets the very poses of the path critic, dwa_planner.cpp:277-281)
  int skip = 0;
};
struct MapGridRobot {  // fleet mode: one per robot, in device memory
  DwaGeom g;
  MapGridJob job[4];
};
struct FleetRobot {
  MapGridRobot grids;  // geometry + the four MapGrid jobs (dist pointers are the robot's distance grids)
  float pos[3], vel[3];
  int osc_mask;
  double scale_alignment;  // 0 once the robot is within forward_point_distance of its goal (dwa_planner.cpp:277-285)
  int nx, ny, nth;
  int samples_offset;  // into the fleet's float sample array: xs | ys | ths of this robot
};

struct MapGridArgs {
  DwaGeom g;  // fleet mode: only sx, sy, res of it are used (shared by all robots)
  int allow_unknown;
  MapGridJob job[4];
  const FleetRobot* fleet;  // null: single planner (g, job above); else CTA b serves robot b / jobs_per_robot
};

constexpr int kMapGridThreads = 512;
constexpr int kMapGridMaxPlanes = 18;

// seeds: plan points from the first one that is on the map and not NO_INFORMATION until the plan first leaves the
// map again (map_grid.cpp:189-202 / :225-239); sets the seed bits in F0 (shared memory, zeroed by the caller).
// Returns false when no plan point is on the map (every cell stays unreachable).
__device__ __forceinline__ bool mapgrid_seed(const MapGridJob& job, const DwaGeom& g, uint32_t* F0, int W) {
  __shared__ int s_first, s_end;
  const int tid = threadIdx.x, nt = blockDim.x;  // (512 threads in the sliced kernels, 32 .. 128 in the row kernel)
  if (tid == 0) {
    s_first = 0x7fffffff;
    s_end = job.n_points;
  }
  __syncthreads();
  // cell of plan point i (my << 16 | mx), or -1 when it is off the map or on NO_INFORMATION.  worldToMap costs two
  // fp64 divisions whenever a point sits on a cell border (plans are often laid out on the grid), so every thread
  // evaluates its points once and keeps the first kCached of them in registers for the later passes.
  constexpr int kCached = 8;
  auto point_cell = [&](int i) -> int {
    int mx, my;
    const double wx = job.plan_xy[2 * i], wy = job.plan_xy[2 * i + 1];
    if (!dwa_world_to_map(g, wx, wy, mx, my)) return -1;
    if (g.cost[(size_t)my * g.pitch + mx] == kNoInfo) return -1;
    return (my << 16) | mx;
  };
  int cached[kCached];
#pragma unroll
  for (int q = 0; q < kCached; ++q) {
    const int i = tid + q * nt;
    cached[q] = i < job.n_points ? point_cell(i) : -1;
    if (cached[q] >= 0) atomicMin(&s_first, i);
  }
  for (int i = tid + kCached * nt; i < job.n_points; i += nt)
    if (point_cell(i) >= 0) atomicMin(&s_first, i);
  __syncthreads();
  const int first = s_first;
  if (first == 0x7fffffff) return false;
#pragma unroll
  for (int q = 0; q < kCached; ++q) {
    const int i = tid + q * nt;
    if (i > first && i < job.n_points && cached[q] < 0) atomicMin(&s_end, i);
  }
  for (int i = tid + kCached * nt; i < job.n_points; i += nt)
    if (i > first && point_cell(i) < 0) atomicMin(&s_end, i);
  __syncthreads();
  const int end = s_end, lo = job.local_goal ? end - 1 : first;
#pragma unroll
  for (int q = 0; q < kCached; ++q) {
    const int i = tid + q * nt;
    if (i >= lo && i < end) atomicOr(&F0[(cached[q] >> 16) * W + ((cached[q] & 0xffff) >> 5)], 1u << (cached[q] & 31));
  }
  for (int i = tid + kCached * nt; i < end; i += nt) {
    if (i < lo) continue;
    const int c = point_cell(i);
    atomicOr(&F0[(c >> 16) * W + ((c & 0xffff) >> 5)], 1u << (c & 31));
  }
  __syncthreads();
  return true;
}

// passable bits of one 32-cell word of the costmap (map_grid.cpp:109-116)
__device__ __forceinline__ uint32_t mapgrid_passable(const DwaGeom& g, int allow_unknown, int r, int w) {
  uint32_t p = 0;
  const uint8_t* row = g.cost + (size_t)r * g.pitch + w * 32;
  const int nbits = min(32, (int)g.sx - w * 32);
  if (nbits == 32 && ((size_t)row & 3) == 0) {
    const uint32_t* row4 = reinterpret_cast<const uint32_t*>(row);
#pragma unroll
    for (int q = 0; q < 8; ++q) {  // four cells per packed compare: obstacle = cost >= 253, minus 255 when unknown is allowed
      const uint32_t v = row4[q];
      const uint32_t ge = __vcmpgeu4(v, 0xfdfdfdfdu);
      const uint32_t obs = allow_unknown ? ge & ~__vcmpeq4(v, 0xffffffffu) : ge;
      const uint32_t bits = ((obs & 0x01010101u) * 0x01020408u) >> 24;  // bit b <-> byte b
      p |= (~bits & 0xfu) << (4 * q);
    }
    return p;
  }
  for (int b = 0; b < nbits; ++b) {
    const uint8_t c = row[b];
    const bool obstacle = c == kLethal || c == kInscribed || (c == kNoInfo && !allow_unknown);
    p |= (uint32_t)(!obstacle) << b;
  }
  return p;
}

// Fast variant: every thread keeps its kWPT words' visited / passable / seed bits and the bit-sliced level counters
// (plane k holds bit k of the level at which each cell was first touched) in REGISTERS; only the frontier goes
// through shared memory, so one level costs five shared loads, a handful of logic ops and one barrier.  After the
// wavefront dies out the planes are parked in shared memory and un-sliced by whole warps (one word per warp step,
// lane = cell) into coalesced uint32 stores.
template <int kWPT>
__global__ void __launch_bounds__(kMapGridThreads, kWPT == 1 ? 2 : 1) k_mapgrid_prepare_sliced(MapGridArgs a, int jobs_per_robot, int planes) {
  extern __shared__ uint32_t mg_smem[];
  cudaTriggerProgrammaticLaunchCompletion();  // the scoring kernel may be scheduled behind us; it waits for our end
  const MapGridJob job = a.fleet ? a.fleet[blockIdx.x / jobs_per_robot].grids.job[blockIdx.x % jobs_per_robot]
                                 : a.job[blockIdx.x % jobs_per_robot];
  if (job.skip) return;
  const DwaGeom g = a.fleet ? a.fleet[blockIdx.x / jobs_per_robot].grids.g : a.g;
  const int W = (g.sx + 31) / 32, NW = W * (int)g.sy;
  uint32_t* F0 = mg_smem;  // NW words + one that stays zero
  uint32_t* F1 = F0 + NW + 1;
  const int tid = threadIdx.x;
  const uint32_t n_cells = g.sx * g.sy;
  if (tid == 0) F0[NW] = F1[NW] = 0;

  uint32_t P[kWPT], V[kWPT], S[kWPT], D[kMapGridMaxPlanes][kWPT];
#pragma unroll
  for (int q = 0; q < kWPT; ++q) {
    const int wi = tid + q * kMapGridThreads;
    P[q] = 0;
    if (wi < NW) {
      P[q] = mapgrid_passable(g, a.allow_unknown, wi / W, wi % W) | (job.within_robot ? job.within_robot[wi] : 0u);
      F0[wi] = 0;
      F1[wi] = 0;
    }
#pragma unroll
    for (int k = 0; k < kMapGridMaxPlanes; ++k) D[k][q] = 0;
  }
  __syncthreads();
  const bool seeded = mapgrid_seed(job, g, F0, W);
#pragma unroll
  for (int q = 0; q < kWPT; ++q) {
    const int wi = tid + q * kMapGridThreads;
    S[q] = (seeded && wi < NW) ? F0[wi] : 0u;
    V[q] = S[q];
  }

  // neighbour word indices and the valid-column mask of every owned word, hoisted out of the level loop; a missing
  // neighbour (map border) reads the always-zero word at index NW
  int iL[kWPT], iR[kWPT], iU[kWPT], iD[kWPT];
  uint32_t colmask[kWPT];
#pragma unroll
  for (int q = 0; q < kWPT; ++q) {
    const int wi = tid + q * kMapGridThreads;
    const int r = wi / W, w = wi - r * W;
    iL[q] = (wi < NW && w > 0) ? wi - 1 : NW;
    iR[q] = (wi < NW && w + 1 < W) ? wi + 1 : NW;
    iU[q] = (wi < NW && r > 0) ? wi - W : NW;
    iD[q] = (wi < NW && r + 1 < (int)g.sy) ? wi + W : NW;
    const int nbits = (int)g.sx - w * 32;
    colmask[q] = wi < NW ? (nbits < 32 ? (1u << nbits) - 1u : 0xffffffffu) : 0u;
  }
  uint32_t last_level = 0;
  if (seeded) {
    // one BFS level: read frontier `F`, write the next one into `Fn`.  Two levels per loop trip with the buffers'
    // roles fixed at compile time, so neighbour loads are [index + constant] and nothing is swapped.
    auto one_level = [&](const uint32_t* F, uint32_t* Fn, uint32_t lv) -> int {
      int any = 0;
#pragma unroll
      for (int q = 0; q < kWPT; ++q) {
        const int wi = tid + q * kMapGridThreads;
        if (kWPT > 1 && wi >= NW) continue;
        const uint32_t f = F[min(wi, NW)];
        const uint32_t nb = ((f << 1) | (f >> 1) | (F[iL[q]] >> 31) | (F[iR[q]] << 31) | F[iU[q]] | F[iD[q]]) & colmask[q];
        const uint32_t touched = nb & ~V[q];
        uint32_t next = 0;
        if (touched) {  // rare: a word is touched during only a few levels
          V[q] |= touched;
          next = touched & P[q];  // obstacles are touched but not expanded (updatePathCell)
          if (next) {
#pragma unroll
            for (int k = 0; k < 8; ++k)
              if ((lv >> k) & 1u) D[k][q] |= next;
            if (lv >> 8) {
#pragma unroll
              for (int k = 8; k < kMapGridMaxPlanes; ++k)
                if ((lv >> k) & 1u) D[k][q] |= next;
            }
          }
        }
        if (wi < NW) Fn[wi] = next;
        any |= next != 0;
      }
      return any;
    };
    // plain barriers between levels; the "anything still moving?" vote only every eighth level (a few empty levels
    // at the end cost less than a reducing barrier per level)
    for (uint32_t level = 0;; level += 8) {
      int any = 0;
#pragma unroll
      for (uint32_t s2 = 0; s2 < 8; s2 += 2) {
        any |= one_level(F0, F1, level + s2 + 1);
        __syncthreads();
        any |= one_level(F1, F0, level + s2 + 2);
        if (s2 < 6) __syncthreads();
      }
      last_level = level + 8;
      if (!__syncthreads_or(any)) break;
    }
  }
  __syncthreads();
  planes = min(planes, 32 - __clz(last_level));  // only the planes the deepest level reached can hold a set bit
  // park V, P, S and the planes: layout [3 + planes][NW]
  uint32_t* park = mg_smem;
#pragma unroll
  for (int q = 0; q < kWPT; ++q) {
    const int wi = tid + q * kMapGridThreads;
    if (wi >= NW) continue;
    park[wi] = V[q];
    park[NW + wi] = P[q];
    park[2 * NW + wi] = S[q];
#pragma unroll
    for (int k = 0; k < kMapGridMaxPlanes; ++k)
      if (k < planes) park[(3 + k) * NW + wi] = D[k][q];
  }
  __syncthreads();
  const int lane = tid & 31, warp = tid >> 5;
  for (int r = warp; r < (int)g.sy; r += kMapGridThreads / 32) {  // a warp per row, a lane per cell of each word
    for (int w = 0; w < W; ++w) {
      const int wi = r * W + w, c = w * 32 + lane;
      // un-slice: lane k loads plane k of this word; a 32 x 32 bit transpose across the warp (five butterfly steps)
      // leaves in lane j the word whose bit k is bit j of plane k, i.e. the level of cell j
      uint32_t d = lane < planes ? park[(3 + lane) * NW + wi] : 0u;
#pragma unroll
      for (int sft = 16; sft > 0; sft >>= 1) {
        const uint32_t keep_lo = sft == 16 ? 0x0000ffffu : sft == 8 ? 0x00ff00ffu : sft == 4 ? 0x0f0f0f0fu : sft == 2 ? 0x33333333u : 0x55555555u;
        const uint32_t other = __shfl_xor_sync(0xffffffffu, d, sft);
        d = (lane & sft) ? ((d & ~keep_lo) | ((other & ~keep_lo) >> sft)) : ((d & keep_lo) | ((other & keep_lo) << sft));
      }
      if (c >= (int)g.sx) continue;
      const uint32_t v = (park[wi] >> lane) & 1u, p = (park[NW + wi] >> lane) & 1u, sd = (park[2 * NW + wi] >> lane) & 1u;
      // seeds 0 (even on an obstacle), untouched cells unreachableCellCosts, touched obstacles obstacleCosts
      job.dist[(size_t)r * g.sx + c] = sd ? 0u : (!v ? n_cells + 1 : (!p ? n_cells : d));
    }
  }
}

// Row variant for local maps of at most 128 x 128 cells (the usual 6 m window is 120 x 120): NO barrier and NO shared
// memory inside a level.  A lane of a search warp owns kRPL consecutive rows of 4 words (128 cells) each -- frontier,
// "passable and not yet visited" bits and the eight low bit planes of the level all live in its registers; the row
// above / below the lane's rows comes through two warp shuffles per word, the left / right cell through funnel shifts:
//     next = (F<<1 | F>>1 | F(up) | F(down)) & A;   A ^= next;   low planes |= next by the level's (static) low bits
// and once per kTrip levels the planes above take T = A(before) ^ A(after) by the bits those levels share: ~7
// instructions per word and level against five shared loads, a store and a CTA barrier in the sliced kernel.
// Search warp w owns rows [w * own, (w + 1) * own) and carries `halo` more rows on either side; rows at distance t from
// the window's edge go stale after t levels (their outer neighbours are missing), so the warps run `halo` levels on
// their own, then publish their own rows (F, A) in shared memory and refresh their halo rows: one (named) barrier per
// `halo` levels -- 16 at 120 rows and 4 warps -- instead of one per level.
// Touched-but-not-expanded cells (obstacles next to an expanded cell) are derived once at the end as the neighbours
// of the expanded set, instead of being tracked per level.  Levels >= 256 (mazes) leave the planes: those cells are
// written to the grid as they are reached and flagged in a ninth plane (shared memory), which the epilogue skips.
// A planner's launch has 512 threads: the warps beyond the search warps compute passable bits and seeds with them,
// sleep at the CTA barrier during the search and share the epilogue (planes parked in shared memory; four cells per
// lane spread into the bytes of one word by nibble * 0x204081 & 0x01010101; uint4 stores).  A fleet's launch has the
// search warps only (thousands of grids: occupancy instead of latency).
// Measured (C2, 144 levels): 42 us sliced -> 28 us; the search is bound by the ALU pipe of the four schedulers (one
// warp instruction per two cycles each, B300_MICROARCH "pipe rates"), ~55 instructions per level and warp.
template <int kWarps, int kRPL, int kTrip>
__global__ void __launch_bounds__(512) k_mapgrid_prepare_rows(MapGridArgs a, int jobs_per_robot) {
  extern __shared__ uint32_t mg_smem[];
  cudaTriggerProgrammaticLaunchCompletion();  // the scoring kernel may be scheduled behind us; it waits for our end
  const MapGridJob job = a.fleet ? a.fleet[blockIdx.x / jobs_per_robot].grids.job[blockIdx.x % jobs_per_robot]
                                 : a.job[blockIdx.x % jobs_per_robot];
  if (job.skip) return;
  const DwaGeom g = a.fleet ? a.fleet[blockIdx.x / jobs_per_robot].grids.g : a.g;
  static_assert(kWarps > 1 && (kTrip == 4 || kTrip == 8), "search warps exchange halo rows; trips of 4 or 8 levels");
  constexpr int kWin = 32 * kRPL, kSearchThreads = 32 * kWarps;
  constexpr uint32_t kFull = 0xffffffffu;
  const int nt = blockDim.x;  // 32 * kWarps, or 512: the extra warps help before and after the search
  const int W = (g.sx + 31) / 32, sy = (int)g.sy, NW = W * sy;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t n_cells = g.sx * g.sy;
  uint32_t* Psm = mg_smem;      // passable bits, [row][W]
  uint32_t* Ssm = Psm + NW;     // seed bits
  uint32_t* Dsm = Ssm + NW;     // cells of level >= 256 (written to the grid as they were reached)
  uint32_t* XF = Dsm + NW;      // published rows, two buffers of F | A; the touched bits at the end
  uint32_t* Pl = XF + 4 * NW;   // the eight planes, parked for the epilogue
  for (int wi = tid; wi < NW; wi += nt) {
    Psm[wi] = mapgrid_passable(g, a.allow_unknown, wi / W, wi % W) | (job.within_robot ? job.within_robot[wi] : 0u);
    Ssm[wi] = 0;
    Dsm[wi] = 0;
  }
  __syncthreads();
  mapgrid_seed(job, g, Ssm, W);  // (no seed: every bit stays 0, every cell unreachable)

  if (warp < kWarps) {  // ---- the search, by the first kWarps warps (barrier 1 is theirs; the others wait below)
  auto search_barrier_or = [&](bool pred) -> bool {
    uint32_t r;
    asm volatile("{ .reg .pred p, q; setp.ne.u32 q, %1, 0; bar.red.or.pred p, 1, %2, q; selp.u32 %0, 1, 0, p; }"
                 : "=r"(r) : "r"((uint32_t)pred), "n"(kSearchThreads) : "memory");
    return r != 0;
  };
  // rows of this lane: row0 + j; own rows of the warp [own_lo, own_hi).  The first row of lane 0 and the last row of
  // lane 31 are never rows whose bits matter (off the map, or the outermost halo rows), so the shuffles at the warp's
  // ends need no masking: whatever they deliver lands in rows that are empty or stale by design.
  const int own = (sy + kWarps - 1) / kWarps;
  const int margin = (kWin - own) / 2;
  const int halo = margin & ~7;  // levels between exchanges (>= 8 for every map the host sends here)
  const int own_lo = warp * own, own_hi = min(own_lo + own, sy);
  const int row0 = own_lo - margin + lane * kRPL;
  uint32_t F[kRPL][4], G[kRPL][4], A[kRPL][4], T[kRPL][4], D[8][kRPL][4];
#pragma unroll
  for (int j = 0; j < kRPL; ++j)
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const int r = row0 + j;
      const bool in = r >= 0 && r < sy && w < W;
      const uint32_t p = in ? Psm[r * W + w] : 0u, sd = in ? Ssm[r * W + w] : 0u;
      F[j][w] = sd;
      A[j][w] = p & ~sd;
#pragma unroll
      for (int k = 0; k < 8; ++k) D[k][j][w] = 0;
    }
  // the four neighbours of the bits of X, into Y (every row of the window; the outermost rows get whatever the
  // shuffle delivers at the warp's ends)
  auto neighbours = [&](const uint32_t (&X)[kRPL][4], uint32_t (&Y)[kRPL][4]) {
    uint32_t up[4], dn[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      up[w] = __shfl_up_sync(kFull, X[kRPL - 1][w], 1);
      dn[w] = __shfl_down_sync(kFull, X[0][w], 1);
    }
#pragma unroll
    for (int j = 0; j < kRPL; ++j)
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        const uint32_t f = X[j][w], l = w ? X[j][w - 1] : 0u, r = w < 3 ? X[j][w + 1] : 0u;
        const uint32_t u = j ? X[j - 1][w] : up[w], d = j < kRPL - 1 ? X[j + 1][w] : dn[w];
        Y[j][w] = __funnelshift_l(l, f, 1) | __funnelshift_r(f, r, 1) | u | d;
      }
  };
  // level `base + i` (i < kTrip at compile time): the low planes take the new cells of the levels whose bit is set.
  // kDeep (levels >= 256, a maze: rare) is a separate instantiation so that the usual loop stays a few hundred
  // instructions of straight-line code -- a lone warp per scheduler has nothing to hide instruction fetches behind.
  auto one_level = [&](const uint32_t (&X)[kRPL][4], uint32_t (&Y)[kRPL][4], uint32_t base, auto ic, auto deep) {
    constexpr int i = decltype(ic)::value;
    neighbours(X, Y);
#pragma unroll
    for (int j = 0; j < kRPL; ++j)
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        Y[j][w] &= A[j][w];
        A[j][w] ^= Y[j][w];
        if (i & 1) D[0][j][w] |= Y[j][w];
        if (i & 2) D[1][j][w] |= Y[j][w];
        if (i & 4) D[2][j][w] |= Y[j][w];
      }
    if (decltype(deep)::value) {  // the level no longer fits the planes: the cells are written as they are reached
#pragma unroll 1
      for (int j = 0; j < kRPL; ++j) {
        const int r = row0 + j;
        if (r < own_lo || r >= own_hi) continue;
#pragma unroll 1
        for (int w = 0; w < W; ++w) {
          uint32_t m = 0;
#pragma unroll
          for (int jj = 0; jj < kRPL; ++jj)
#pragma unroll
            for (int ww = 0; ww < 4; ++ww)
              if (jj == j && ww == w) m = Y[jj][ww];
          if (m) Dsm[r * W + w] |= m;  // (the word belongs to this lane)
          while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            job.dist[(size_t)r * g.sx + w * 32 + b] = base + i;
          }
        }
      }
    }
  };
  // levels base .. base + kTrip - 1 (base a multiple of kTrip): the cells reached in them share the level's bits from
  // log2(kTrip) up, which are set once per trip from T = A(before) ^ A(after)
  auto trip = [&](uint32_t base, auto deep) {
#pragma unroll
    for (int j = 0; j < kRPL; ++j)
#pragma unroll
      for (int w = 0; w < 4; ++w) T[j][w] = A[j][w];
    if (base) one_level(F, G, base, std::integral_constant<int, 0>(), deep);  // (level 0 is the seeds themselves)
    else {
#pragma unroll
      for (int j = 0; j < kRPL; ++j)
#pragma unroll
        for (int w = 0; w < 4; ++w) G[j][w] = F[j][w];
    }
    one_level(G, F, base, std::integral_constant<int, 1>(), deep);
    one_level(F, G, base, std::integral_constant<int, 2>(), deep);
    one_level(G, F, base, std::integral_constant<int, 3>(), deep);
    if (kTrip == 8) {
      one_level(F, G, base, std::integral_constant<int, 4>(), deep);
      one_level(G, F, base, std::integral_constant<int, 5>(), deep);
      one_level(F, G, base, std::integral_constant<int, 6>(), deep);
      one_level(G, F, base, std::integral_constant<int, 7>(), deep);
    }
#pragma unroll
    for (int j = 0; j < kRPL; ++j)
#pragma unroll
      for (int w = 0; w < 4; ++w) T[j][w] ^= A[j][w];
#pragma unroll
    for (int k = (kTrip == 8 ? 3 : 2); k < 8; ++k)
      if ((base >> k) & 1u) {
#pragma unroll
        for (int j = 0; j < kRPL; ++j)
#pragma unroll
          for (int w = 0; w < 4; ++w) D[k][j][w] |= T[j][w];
      }
  };
  auto trips = [&](uint32_t base) {
    if (base < 256) trip(base, std::false_type());
    else trip(base, std::true_type());
  };
  auto own_rows_or = [&](const uint32_t (&X)[kRPL][4]) -> uint32_t {
    uint32_t any = 0;
#pragma unroll
    for (int j = 0; j < kRPL; ++j) {
      const int r = row0 + j;
      if (r >= own_lo && r < own_hi) any |= X[j][0] | X[j][1] | X[j][2] | X[j][3];
    }
    return any;
  };
  // publish the own rows of X / refresh the rows of the window that other warps own
  auto publish = [&](uint32_t* buf, const uint32_t (&X)[kRPL][4]) {
#pragma unroll
    for (int j = 0; j < kRPL; ++j) {
      const int r = row0 + j;
      if (r < own_lo || r >= own_hi) continue;
#pragma unroll
      for (int w = 0; w < 4; ++w)
        if (w < W) buf[r * W + w] = X[j][w];
    }
  };
  auto refresh = [&](const uint32_t* buf, uint32_t (&X)[kRPL][4]) {
#pragma unroll
    for (int j = 0; j < kRPL; ++j) {
      const int r = row0 + j;
      if (r < 0 || r >= sy || (r >= own_lo && r < own_hi)) continue;
#pragma unroll
      for (int w = 0; w < 4; ++w)
        if (w < W) X[j][w] = buf[r * W + w];
    }
  };

  uint32_t lv = 0;  // levels done (a multiple of kTrip); the frontier of level lv - 1 (the seeds at first) is in F
  {
    for (uint32_t e = 0;; ++e) {
#pragma unroll 1
      for (int t = 0; t < halo; t += kTrip) {
        trips(lv);
        lv += kTrip;
      }
      uint32_t* buf = XF + (e & 1u) * 2 * NW;
      publish(buf, F);
      publish(buf + NW, A);
      if (!search_barrier_or(own_rows_or(F) != 0)) break;  // exact rows only: an empty frontier everywhere ends the search
      refresh(buf, F);
      refresh(buf + NW, A);
    }
  }

  // expanded cells E = seeds | visited passable cells; touched = E | neighbours(E)
#pragma unroll
  for (int j = 0; j < kRPL; ++j)
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const int r = row0 + j;
      const bool in = r >= 0 && r < sy && w < W;
      F[j][w] = in ? (Ssm[r * W + w] | (Psm[r * W + w] & ~A[j][w])) : 0u;
    }
  search_barrier_or(false);  // (everyone has left the loop: the exchange buffers are free)
  publish(XF, F);
  search_barrier_or(false);
  refresh(XF, F);
  search_barrier_or(false);  // (... and read, before the touched bits overwrite them)
  neighbours(F, G);
  // park what the epilogue needs of the own rows: touched bits and the planes
#pragma unroll
  for (int j = 0; j < kRPL; ++j) {
    const int r = row0 + j;
    if (r < own_lo || r >= own_hi) continue;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      if (w >= W) continue;
      XF[r * W + w] = F[j][w] | G[j][w];
#pragma unroll
      for (int k = 0; k < 8; ++k) Pl[k * NW + r * W + w] = D[k][j][w];
    }
  }
  }  // ---- end of the search warps' part
  __syncthreads();
  // Epilogue, every warp of the CTA: a warp per row, a lane per four cells.  The planes of four cells are spread into
  // the bytes of one word (nibble * 0x204081 & 0x01010101 puts bit b into byte b); seeds 0 (even on an obstacle),
  // untouched cells unreachableCellCosts, touched obstacles obstacleCosts; uint4 stores.
  const bool vec = (g.sx & 3u) == 0 && ((size_t)job.dist & 15u) == 0;
  const int w = lane >> 3, c = (lane & 7) * 4;
  const int ncols = min(32, (int)g.sx - w * 32);
  for (int r = warp; r < sy; r += nt >> 5) {
    if (w >= W || c >= ncols) continue;
    const int wi = r * W + w;
    const uint32_t touched = XF[wi], pw = Psm[wi], sw = Ssm[wi];
    const uint32_t unreached = ~touched >> c, obstacle = (touched & ~pw & ~sw) >> c, seed = sw >> c;
    const uint32_t dn = (Dsm[wi] >> c) & 0xfu;  // cells written during the search keep their value
    uint32_t lo = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) lo |= ((((Pl[k * NW + wi] >> c) & 0xfu) * 0x00204081u) & 0x01010101u) << k;
    uint32_t out[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      uint32_t v = (lo >> (8 * b)) & 0xffu;
      v = ((seed >> b) & 1u) ? 0u : v;
      v = ((obstacle >> b) & 1u) ? n_cells : v;
      v = ((unreached >> b) & 1u) ? n_cells + 1 : v;
      out[b] = v;
    }
    uint32_t* dst = job.dist + (size_t)r * g.sx + w * 32 + c;
    if (vec && dn == 0) {
      *reinterpret_cast<uint4*>(dst) = make_uint4(out[0], out[1], out[2], out[3]);
    } else {
#pragma unroll
      for (int b = 0; b < 4; ++b)
        if (c + b < ncols && !((dn >> b) & 1u)) dst[b] = out[b];
    }
  }
}

// General variant for local costmaps too large for the register-resident kernel: all bit planes in shared memory,
// distances written as cells are touched.
__global__ void __launch_bounds__(kMapGridThreads) k_mapgrid_prepare(MapGridArgs a, int jobs_per_robot) {
  extern __shared__ uint32_t mg_smem[];
  const MapGridJob job = a.fleet ? a.fleet[blockIdx.x / jobs_per_robot].grids.job[blockIdx.x % jobs_per_robot]
                                 : a.job[blockIdx.x % jobs_per_robot];
  if (job.skip) return;
  const DwaGeom g = a.fleet ? a.fleet[blockIdx.x / jobs_per_robot].grids.g : a.g;
  const int W = (g.sx + 31) / 32, NW = W * (int)g.sy;
  uint32_t* P = mg_smem;
  uint32_t* V = P + NW;
  uint32_t* F0 = V + NW;
  uint32_t* F1 = F0 + NW;
  __shared__ int s_first, s_end;
  const int tid = threadIdx.x;
  const uint32_t n_cells = g.sx * g.sy;

  for (uint32_t i = tid; i < n_cells; i += kMapGridThreads) job.dist[i] = n_cells + 1;  // resetPathDist
  for (int wi = tid; wi < NW; wi += kMapGridThreads) {
    const int r = wi / W, w = wi - r * W;
    uint32_t p = 0;
    const uint8_t* row = g.cost + (size_t)r * g.pitch + w * 32;
    const int nbits = min(32, (int)g.sx - w * 32);
    for (int b = 0; b < nbits; ++b) {
      const uint8_t c = row[b];
      const bool obstacle = c == kLethal || c == kInscribed || (c == kNoInfo && !a.allow_unknown);  // map_grid.cpp:109-116
      p |= (uint32_t)(!obstacle) << b;
    }
    P[wi] = p | (job.within_robot ? job.within_robot[wi] : 0u);
    V[wi] = 0;
    F0[wi] = 0;
    F1[wi] = 0;
  }
  if (tid == 0) {
    s_first = 0x7fffffff;
    s_end = job.n_points;
  }
  __syncthreads();

  // seeds: plan points from the first one that is on the map and not NO_INFORMATION until the plan first leaves the
  // map again (map_grid.cpp:189-202 / :225-239)
  auto point_ok = [&](int i, int& mx, int& my) -> bool {
    const double wx = job.plan_xy[2 * i], wy = job.plan_xy[2 * i + 1];
    if (!dwa_world_to_map(g, wx, wy, mx, my)) return false;
    return g.cost[(size_t)my * g.pitch + mx] != kNoInfo;
  };
  for (int i = tid; i < job.n_points; i += kMapGridThreads) {
    int mx, my;
    if (point_ok(i, mx, my)) atomicMin(&s_first, i);
  }
  __syncthreads();
  const int first = s_first;
  if (first == 0x7fffffff) return;  // nothing on the map: every cell stays unreachable
  for (int i = first + 1 + tid; i < job.n_points; i += kMapGridThreads) {
    int mx, my;
    if (!point_ok(i, mx, my)) atomicMin(&s_end, i);
  }
  __syncthreads();
  const int end = s_end;
  for (int i = (job.local_goal ? end - 1 : first) + tid; i < end; i += kMapGridThreads) {
    int mx, my;
    point_ok(i, mx, my);
    const int wi = my * W + (mx >> 5);
    atomicOr(&F0[wi], 1u << (mx & 31));
    atomicOr(&V[wi], 1u << (mx & 31));
    job.dist[(size_t)my * g.sx + mx] = 0;
  }
  __syncthreads();

  uint32_t* F = F0;
  uint32_t* Fn = F1;
  for (uint32_t level = 0;; ++level) {
    int any = 0;
    for (int wi = tid; wi < NW; wi += kMapGridThreads) {
      const int r = wi / W, w = wi - r * W;
      const uint32_t f = F[wi];
      uint32_t nb = (f << 1) | (f >> 1);
      if (w > 0) nb |= F[wi - 1] >> 31;
      if (w + 1 < W) nb |= F[wi + 1] << 31;
      if (r > 0) nb |= F[wi - W];
      if (r + 1 < (int)g.sy) nb |= F[wi + W];
      const int nbits = (int)g.sx - w * 32;
      if (nbits < 32) nb &= (1u << nbits) - 1u;
      const uint32_t v = V[wi];
      const uint32_t touched = nb & ~v;
      uint32_t next = 0;
      if (touched) {
        V[wi] = v | touched;
        const uint32_t p = P[wi];
        next = touched & p;
        uint32_t t = touched;
        uint32_t* drow = job.dist + (size_t)r * g.sx + w * 32;
        while (t) {
          const int b = __ffs(t) - 1;
          t &= t - 1;
          drow[b] = ((p >> b) & 1u) ? level + 1 : n_cells;
        }
      }
      Fn[wi] = next;
      any |= next != 0;
    }
    if (!__syncthreads_or(any)) break;
    uint32_t* tmp = F;
    F = Fn;
    Fn = tmp;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Rollout + the six critics + argmin: SimpleTrajectoryGenerator::generateTrajectory
// (base_local_planner/src/simple_trajectory_generator.cpp:180-276), OscillationCostFunction::scoreTrajectory
// (src/oscillation_cost_function.cpp:166-176), ObstacleCostFunction::scoreTrajectory + CostmapModel::footprintCost
// (src/obstacle_cost_function.cpp:74-142, src/costmap_model.cpp:50-142, include/base_local_planner/world_model.h:65-86,
// line_iterator.h:38-139), MapGridCostFunction::scoreTrajectory (src/map_grid_cost_function.cpp:75-129) and
// SimpleScoredSamplingPlanner::scoreTrajectory/findBestTrajectory (src/simple_scored_sampling_planner.cpp:50-142).
//
// One warp per velocity sample, one lane per trajectory point.  The float32 Euler state is a sequential recurrence
// (every step rounds to float), but its trig terms depend only on the heading sequence, which is a cheap scalar
// recurrence: all lanes replay theta, each lane evaluates cos/sin for its own step in fp64, and the x/y prefix is
// accumulated with shuffles in the reference's order and rounding.  No FMA contraction (-fmad=false).
// Result record of one search, written by the finishing step
struct DwaDeviceResult {
  double cost, xv, yv, thetav;
  long long best_index;
  int n_points, n_scored;
};

// ---------------------------------------------------------------------------------------------------------------
// A planner's per-cycle scalar arithmetic, shared by the host (navgpu_dwa_*, navgpu_fleet_step) and the device fleet
// step (k_fleet_prepare, k_fleet_apply): IEEE operations without a libm call, compiled with -fmad=false on both sides,
// so both give the same bits.  (std::min / std::max restated: a < b picks as they do, for device code.)
__host__ __device__ inline double dwa_min(double a, double b) { return b < a ? b : a; }
__host__ __device__ inline double dwa_max(double a, double b) { return a < b ? b : a; }

// the most samples VelocityIterator gives an axis configured with n (>= 1) samples: max(2, n) - 1 steps, the zero it
// inserts once when the range crosses it, and the maximum
__host__ __device__ inline int dwa_axis_bound(int n) { return (n < 2 ? 2 : n) + 1; }

// VelocityIterator, base_local_planner/include/base_local_planner/velocity_iterator.h:49-74: the samples of [mn, mx]
// as floats into out (room for dwa_axis_bound(n)); returns how many
__host__ __device__ inline int velocity_samples(double mn, double mx, int n, float* out) {
  if (mn == mx) {
    out[0] = (float)mn;
    return 1;
  }
  n = n < 2 ? 2 : n;
  const double step = (mx - mn) / double(n - 1 < 1 ? 1 : n - 1);
  double cur, next = mn;
  int k = 0;
  for (int j = 0; j < n - 1; ++j) {
    cur = next;
    next += step;
    out[k++] = (float)cur;
    if (cur < 0 && next > 0) out[k++] = 0.0f;
  }
  out[k++] = (float)mx;
  return k;
}

// the per-axis sample counts of the configuration (dwa_planner.cpp:86-109) and their bounds
__host__ __device__ inline void dwa_axis_samples(const navgpu_dwa_config& cfg, int n[3]) {
  n[0] = cfg.vx_samples <= 0 ? 1 : cfg.vx_samples;
  n[1] = cfg.vy_samples <= 0 ? 1 : cfg.vy_samples;
  n[2] = cfg.vth_samples <= 0 ? 1 : cfg.vth_samples;
}

// SimpleTrajectoryGenerator::initialise, simple_trajectory_generator.cpp:60-135: xs | ys | ths into out (room for the
// three dwa_axis_bound), their counts into counts.  The use_dwa = 0 window takes hypot, which only the host may call
// for bit-exact results: the device fleet step refuses such configurations.
__host__ __device__ inline void enumerate_samples(const navgpu_dwa_config& cfg, const float pos[3], const float vel[3],
                                                  const float goal[2], float* out, int counts[3]) {
  const double max_vel_th = cfg.max_rot_vel, min_vel_th = -1.0 * max_vel_th;
  const float acc[3] = {float(cfg.acc_lim_x), float(cfg.acc_lim_y), float(cfg.acc_lim_theta)};
  double min_vel_x = cfg.min_vel_x, max_vel_x = cfg.max_vel_x, min_vel_y = cfg.min_vel_y, max_vel_y = cfg.max_vel_y;
  int n[3];
  dwa_axis_samples(cfg, n);
  float mx[3], mn[3];
  if (!cfg.use_dwa) {
    const double dist = hypot(goal[0] - pos[0], goal[1] - pos[1]);
    max_vel_x = dwa_max(dwa_min(max_vel_x, dist / cfg.sim_time), min_vel_x);
    max_vel_y = dwa_max(dwa_min(max_vel_y, dist / cfg.sim_time), min_vel_y);
    mx[0] = dwa_min(max_vel_x, vel[0] + acc[0] * cfg.sim_time);
    mx[1] = dwa_min(max_vel_y, vel[1] + acc[1] * cfg.sim_time);
    mx[2] = dwa_min(max_vel_th, vel[2] + acc[2] * cfg.sim_time);
    mn[0] = dwa_max(min_vel_x, vel[0] - acc[0] * cfg.sim_time);
    mn[1] = dwa_max(min_vel_y, vel[1] - acc[1] * cfg.sim_time);
    mn[2] = dwa_max(min_vel_th, vel[2] - acc[2] * cfg.sim_time);
  } else {
    mx[0] = dwa_min(max_vel_x, vel[0] + acc[0] * cfg.sim_period);
    mx[1] = dwa_min(max_vel_y, vel[1] + acc[1] * cfg.sim_period);
    mx[2] = dwa_min(max_vel_th, vel[2] + acc[2] * cfg.sim_period);
    mn[0] = dwa_max(min_vel_x, vel[0] - acc[0] * cfg.sim_period);
    mn[1] = dwa_max(min_vel_y, vel[1] - acc[1] * cfg.sim_period);
    mn[2] = dwa_max(min_vel_th, vel[2] - acc[2] * cfg.sim_period);
  }
  int k = 0;
  for (int a = 0; a < 3; ++a) {
    counts[a] = velocity_samples(mn[a], mx[a], n[a], out + k);
    k += counts[a];
  }
}

// OscillationCostFunction's latched state (oscillation_cost_function.h:78-83, .cpp:56-164)
struct Oscillation {
  bool strafe_pos_only = false, strafe_neg_only = false, strafing_pos = false, strafing_neg = false;
  bool rot_pos_only = false, rot_neg_only = false, rotating_pos = false, rotating_neg = false;
  bool forward_pos_only = false, forward_neg_only = false, forward_pos = false, forward_neg = false;
  float prev[3] = {0.f, 0.f, 0.f};
  __host__ __device__ void reset() {
    strafe_pos_only = strafe_neg_only = strafing_pos = strafing_neg = false;
    rot_pos_only = rot_neg_only = rotating_pos = rotating_neg = false;
    forward_pos_only = forward_neg_only = forward_pos = forward_neg = false;
  }
  __host__ __device__ int mask() const {
    return int(forward_pos_only) | int(forward_neg_only) << 1 | int(strafe_pos_only) << 2 | int(strafe_neg_only) << 3 |
           int(rot_pos_only) << 4 | int(rot_neg_only) << 5;
  }
  __host__ __device__ bool set_flags(double xv, double yv, double thv, double min_vel_trans) {
    bool flag_set = false;
    if (xv < 0.0) { if (forward_pos) { forward_neg_only = true; flag_set = true; } forward_pos = false; forward_neg = true; }
    if (xv > 0.0) { if (forward_neg) { forward_pos_only = true; flag_set = true; } forward_neg = false; forward_pos = true; }
    if (fabs(xv) <= min_vel_trans) {
      if (yv < 0) { if (strafing_pos) { strafe_neg_only = true; flag_set = true; } strafing_pos = false; strafing_neg = true; }
      if (yv > 0) { if (strafing_neg) { strafe_pos_only = true; flag_set = true; } strafing_neg = false; strafing_pos = true; }
      if (thv < 0) { if (rotating_pos) { rot_neg_only = true; flag_set = true; } rotating_pos = false; rotating_neg = true; }
      if (thv > 0) { if (rotating_neg) { rot_pos_only = true; flag_set = true; } rotating_neg = false; rotating_pos = true; }
    }
    return flag_set;
  }
  __host__ __device__ void update(const float pos[3], double cost, double xv, double yv, double thv, double min_vel_trans,
                                  double reset_dist, double reset_angle) {
    if (cost < 0) return;
    if (set_flags(xv, yv, thv, min_vel_trans)) { prev[0] = pos[0]; prev[1] = pos[1]; prev[2] = pos[2]; }
    if (forward_pos_only || forward_neg_only || strafe_pos_only || strafe_neg_only || rot_pos_only || rot_neg_only) {
      const double x_diff = pos[0] - prev[0], y_diff = pos[1] - prev[1];
      const double sq_dist = x_diff * x_diff + y_diff * y_diff;
      const double th_diff = pos[2] - prev[2];
      if (sq_dist > reset_dist * reset_dist || fabs(th_diff) > reset_angle) reset();
    }
  }
};

// what findBestPath does on the host with the winner d of a search (dwa_planner.cpp:316-357): result_traj_'s
// velocities persist across cycles (res_v), then the oscillation flags; fills *out (when given) but its n_points
__host__ __device__ inline void apply_dwa_result(const DwaDeviceResult& d, const navgpu_dwa_config& c, const double pose[3],
                                                 int32_t n_samples, double res_v[3], Oscillation& osc,
                                                 navgpu_dwa_result* out) {
  if (d.cost >= 0) { res_v[0] = d.xv; res_v[1] = d.yv; res_v[2] = d.thetav; }
  const float pos[3] = {(float)pose[0], (float)pose[1], (float)pose[2]};
  // oscillation_costs_.updateOscillationFlags(pos, &result_traj_, min_trans_vel), dwa_planner.cpp:357
  osc.update(pos, d.cost, res_v[0], res_v[1], res_v[2], c.min_trans_vel, c.oscillation_reset_dist,
             c.oscillation_reset_angle);
  if (!out) return;
  out->cost = d.cost;
  out->xv = res_v[0]; out->yv = res_v[1]; out->thetav = res_v[2];
  out->best_index = (int32_t)d.best_index;
  out->n_samples = n_samples;
  out->n_scored = d.n_scored;
}

// What a DWAPlanner fleet keeps per robot from one step to the next: the oscillation flags, result_traj_'s
// velocities, whether a step planned the robot (its distance grids hold that step's wavefronts) and whether its
// alignment grid was its path grid then, and a sensing fleet's rolled origin.  The fleet holds a host and a device
// copy of the array and knows which one is current.
struct FleetDwaState {
  Oscillation osc;
  double res_v[3];
  double origin[2];
  uint8_t planned, aliased;
};

// Multi-GPU sample sweep (config C4): one record per rank and sweep parity in every rank's exchange buffer.  The last
// CTA of a rank's scoring kernel stores its record into EVERY rank's buffer (peer-mapped device memory: the stores
// travel over NVLink), then publishes `seq`; whoever finds all `world` records of the current sweep in its own buffer
// picks the winner.  No host round trip, no collective library call on the path.
constexpr int kShardMaxWorld = 16;
struct ShardSlot {
  double cost;          // the rank's minimum, +inf when it has no valid sample
  long long index;      // its global sample index, -1 when none
  unsigned long long seq;  // sweep number this record belongs to (written last, after a system-wide fence)
  unsigned generated;   // samples the generator accepted on that rank
  unsigned pad_;
};
struct ShardExchange {
  ShardSlot slot[2][kShardMaxWorld];  // [sweep parity][source rank]
};

struct DwaScoreArgs {
  DwaGeom g;
  const uint32_t* dist[4];  // 0 path, 1 goal, 2 goal_front, 3 alignment
  const float* vxs;  // per-axis samples in device memory (only when they do not fit samples_inline)
  const float* vys;
  const float* vths;
  int nx, ny, nth;
  int inline_samples;  // 1: the samples travel in samples_inline (xs | ys | ths), no upload
  float samples_inline[kInlineSamples];
  long long begin, end;  // sample index range scored by this launch
  // block-cyclic sharding of that range: CTA b scores the 8-sample block b * stride_world + stride_rank (1 rank: all)
  int stride_rank, stride_world;
  ShardExchange* shard_peer[kShardMaxWorld];  // every rank's exchange buffer as mapped on this device; null: no exchange
  unsigned long long shard_seq;
  float pos[3], vel[3], acc[3];
  double min_trans_vel, max_trans_vel, min_rot_vel;
  double sim_time, sim_granularity, angular_sim_granularity;
  int use_dwa, sum_scores, allow_unknown, osc_mask;
  double scale_obstacle, scale_goal_front, scale_alignment, scale_path, scale_goal;
  double xshift;
  int nfp;
  double fpx[kMaxFootprint], fpy[kMaxFootprint];
  double* all_terms;   // nullable: 6 doubles per sample of [begin, end): per-critic scaled cost or negative code
  double* block_cost;  // per-CTA minimum
  long long* block_index;
  unsigned int* counters;  // [0] CTAs done, [1] samples the generator accepted
  double* best_cost;       // final (cost, index) of the range; +inf / -1 when none valid
  long long* best_index;
  // when finish_out is set the last CTA also regenerates the winner (findBestTrajectory :123-134) and writes the
  // result record and its points straight into (mapped, pinned) host memory
  DwaDeviceResult* finish_out;
  double* finish_points;
  int finish_capacity;
};

struct TrajResult {
  double cost;  // total per SimpleScoredSamplingPlanner::scoreTrajectory with best_traj_cost = -1 (no early exit)
  bool generated;
  int num_steps;
};

__device__ __forceinline__ double nan_quiet() { return __longlong_as_double(0x7ff8000000000000ll); }

// Map cell (y << 16 | x) of one oriented footprint vertex of one pose, or -1 when it is off the map
// (WorldModel::footprintCost world_model.h:65-86: rotate + translate; CostmapModel::footprintCost worldToMap).
template <class Args>
__device__ __forceinline__ int footprint_vertex_cell(const Args& a, double x, double y, double cos_th, double sin_th,
                                                     int v) {
  const double wx = x + (a.fpx[v] * cos_th - a.fpy[v] * sin_th), wy = y + (a.fpx[v] * sin_th + a.fpy[v] * cos_th);
  int cx, cy;
  if (!dwa_world_to_map(a.g, wx, wy, cx, cy)) return -1;
  return (cy << 16) | cx;
}

// One footprint edge of one pose: CostmapModel::lineCost over the LineIterator cells between the map cells of two
// consecutive oriented footprint vertices (costmap_model.cpp:75-131, line_iterator.h:38-139).  Returns the maximum
// cell cost along the edge, or -1 when a vertex is off the map or a cell is LETHAL / (NO_INFORMATION && !allow_unknown).
// `cost` is the grid the cells are read from: a.g.cost, or the CTA's shared-memory copy of it
template <class Args>
__device__ int footprint_edge_cost(const Args& a, const uint8_t* __restrict__ cost, int cell_p, int cell_q) {
  const DwaGeom& g = a.g;
  if ((cell_p | cell_q) < 0) return -1;  // a vertex off the map (costmap_model.cpp:79-90)
  const int px = cell_p & 0xffff, py = cell_p >> 16, qx = cell_q & 0xffff, qy = cell_q >> 16;
  const int dx = abs(qx - px), dy = abs(qy - py);
  const int xinc = qx >= px ? 1 : -1, yinc = (qy >= py ? 1 : -1) * (int)g.pitch;
  const bool xmajor = dx >= dy;
  const int den = xmajor ? dx : dy, numadd = xmajor ? dy : dx;
  const int major = xmajor ? xinc : yinc, minor = xmajor ? yinc : xinc;
  int num = den / 2;
  int off = py * (int)g.pitch + px;
  // CostmapModel::pointCost (:133-142) rejects LETHAL, and NO_INFORMATION unless unknown cells are allowed; the line
  // cost is the largest cell cost.  Both come out of one running maximum (and, when 255 is allowed, one running
  // minimum of c ^ 0xfe, which is 0 exactly for LETHAL), so the walk costs a load and one or two min/max per cell.
  int best = 0, lethal_probe = 0xff;
  if (a.allow_unknown) {
    for (int k = 0; k <= den; ++k) {
      const int c = cost[off];
      best = max(best, c);
      lethal_probe = min(lethal_probe, c ^ 0xfe);
      num += numadd;
      if (num >= den) {
        num -= den;
        off += minor;
      }
      off += major;
    }
  } else {
    for (int k = 0; k <= den; ++k) {
      best = max(best, (int)cost[off]);
      num += numadd;
      if (num >= den) {
        num -= den;
        off += minor;
      }
      off += major;
    }
  }
  const bool bad = a.allow_unknown ? lethal_probe == 0 : best >= kLethal;
  return bad ? -1 : best;
}
template <class Args>
__device__ __forceinline__ int footprint_edge_cost(const Args& a, int cell_p, int cell_q) {
  return footprint_edge_cost(a, a.g.cost, cell_p, cell_q);
}

// What the critics accumulate over the rounds of 32 points of one trajectory
struct CriticAcc {
  bool obst_fail;
  double obst_sum, obst_last;
  // per map-grid critic: code of the first failing point (0 = none yet) and the value at the last point
  double grid_code[4], grid_last[4];
};
__device__ __forceinline__ void critic_acc_init(CriticAcc& acc) {
  acc.obst_fail = false;
  acc.obst_sum = acc.obst_last = 0.0;
#pragma unroll
  for (int k = 0; k < 4; ++k) acc.grid_code[k] = acc.grid_last[k] = 0.0;
}

// The obstacle critic and the four map-grid critics on one round of up to 32 trajectory points: lane l < cnt holds
// point l -- world position (px, py) and cos / sin of its heading (obstacle_cost_function.cpp:74-142,
// map_grid_cost_function.cpp:75-129).  Shared by the sample sweep (the points come out of the rollout) and by the
// TrajectoryCostFunction backend (the points come from the caller's Trajectory).
__device__ __forceinline__ void score_round(const DwaScoreArgs& a, const uint8_t* __restrict__ cost, int lane, int cnt,
                                            double px, double py, double c, double s, double* warp_scratch,
                                            CriticAcc& acc) {
  const bool active = lane < cnt;
  // ---- obstacle critic: (point, edge) work items spread over all 32 lanes, so a short tail round costs one edge
  // per lane instead of a whole footprint per active lane
  double* pose_s = warp_scratch;              // x, y, cos, sin of the round's points
  // per point: max edge cost; bit 31 set (the unsigned maximum) once any edge of the point is illegal
  unsigned* edge_max = reinterpret_cast<unsigned*>(warp_scratch + 128);
  pose_s[lane] = px;
  pose_s[32 + lane] = py;
  pose_s[64 + lane] = c;
  pose_s[96 + lane] = s;
  edge_max[lane] = 0;
  __syncwarp();
  double occ = 0.0;
  bool fail = false;
  if (a.nfp >= 3) {
    // every (point, vertex) cell once, then every (point, edge) walk between two of them
    // [point][vertex], packed with a row length of nfp: item `it` of the loops below owns word `it`, so the lanes of
    // a pass read and write 32 consecutive words (a row length of kMaxFootprint = 16 put every second point on the
    // same banks)
    int* vcell = reinterpret_cast<int*>(warp_scratch + 128 + 16);
    const int items = cnt * a.nfp;
    // it / nfp for it < 512, nfp <= 16 as a multiply by ceil(2^16 / nfp) (error < 512 / 2^16 < 1 / nfp: exact)
    const unsigned inv_nfp = (65536u + (unsigned)a.nfp - 1u) / (unsigned)a.nfp;
    for (int it = lane; it < items; it += 32) {
      const int p = (int)(((unsigned)it * inv_nfp) >> 16), v = it - p * a.nfp;
      vcell[it] = footprint_vertex_cell(a, pose_s[p], pose_s[32 + p], pose_s[64 + p], pose_s[96 + p], v);
    }
    __syncwarp();
    for (int it = lane; it < items; it += 32) {
      const int p = (int)(((unsigned)it * inv_nfp) >> 16), e = it - p * a.nfp;
      const int next = e + 1 < a.nfp ? it + 1 : it - e;  // the closing edge returns to the point's first vertex
      const int ec = footprint_edge_cost(a, cost, vcell[it], vcell[next]);
      atomicMax(&edge_max[p], ec < 0 ? 0x80000000u : (unsigned)ec);
    }
    __syncwarp();
  }
  // the cell of the point itself serves the obstacle critic's centre lookup and the path / goal grids; the point
  // shifted ahead by xshift serves goal_front / alignment: two worldToMap per point instead of five
  int cell0_x = 0, cell0_y = 0, cell1_x = 0, cell1_y = 0;
  bool on_map0 = false, on_map1 = false;
  if (active) {
    on_map0 = dwa_world_to_map(a.g, px, py, cell0_x, cell0_y);
    if (a.xshift != 0.0) {
      on_map1 = dwa_world_to_map(a.g, px + a.xshift * c, py + a.xshift * s, cell1_x, cell1_y);
    } else {
      on_map1 = on_map0; cell1_x = cell0_x; cell1_y = cell0_y;
    }
  }
  if (active) {
    const int cx = cell0_x, cy = cell0_y;
    if (a.nfp == 0 || !on_map0) fail = true;  // off-map centre: costmap_model.cpp:57-58
    else {
      const int centre = cost[cy * (int)a.g.pitch + cx];
      int f = (int)edge_max[lane];
      if (a.nfp < 3) {  // point robot: the centre cell alone (:61-67)
        f = (centre == kLethal || centre == kInscribed || (centre == kNoInfo && !a.allow_unknown)) ? -1 : centre;
      }
      if (f < 0) fail = true;
      else occ = fmax(fmax(0.0, (double)f), (double)centre);
    }
  }
  acc.obst_fail |= __any_sync(0xffffffffu, fail);
  double ssum = occ;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ssum += __shfl_xor_sync(0xffffffffu, ssum, o);  // small integers: exact
  acc.obst_sum += ssum;
  acc.obst_last = __shfl_sync(0xffffffffu, occ, cnt - 1);
  __syncwarp();
  // ---- the four map-grid critics on my point (the grids come from the kernel launched before this one)
  cudaGridDependencySynchronize();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const bool shifted = k >= 2;        // goal_front, alignment use xshift (dwa_planner.cpp:80-81)
    const bool stop_on_failure = k < 2;  // path, goal (:126-127 turn it off for the other two)
    double code = 0.0, d = 0.0;
    if (active) {
      const int cx = shifted ? cell1_x : cell0_x, cy = shifted ? cell1_y : cell0_y;
      if (!(shifted ? on_map1 : on_map0)) code = -4.0;
      else {
        const uint32_t dd = a.dist[k][cy * (int)a.g.sx + cx];
        const uint32_t n_cells = a.g.sx * a.g.sy;
        d = (double)dd;
        if (stop_on_failure) {
          if (dd == n_cells) code = -3.0;
          else if (dd == n_cells + 1) code = -2.0;
        }
      }
    }
    const unsigned failing = __ballot_sync(0xffffffffu, code != 0.0);
    if (failing && acc.grid_code[k] == 0.0) acc.grid_code[k] = __shfl_sync(0xffffffffu, code, __ffs(failing) - 1);
    acc.grid_last[k] = __shfl_sync(0xffffffffu, d, cnt - 1);
  }
}

// SimpleScoredSamplingPlanner::scoreTrajectory with critics in DWAPlanner's order (dwa_planner.cpp:167-173): the
// total of one trajectory from what the critics found; terms_out (nullable, lane 0 writes) receives the six terms.
__device__ __forceinline__ double combine_critics(const DwaScoreArgs& a, bool osc_bad, const CriticAcc& acc, double* terms_out,
                                                  int lane) {
  const double raw[6] = {osc_bad ? -5.0 : 0.0,
                         a.nfp == 0 ? -9.0 : (acc.obst_fail ? -6.0 : (a.sum_scores ? acc.obst_sum : acc.obst_last)),
                         acc.grid_code[2] != 0.0 ? acc.grid_code[2] : acc.grid_last[2],
                         acc.grid_code[3] != 0.0 ? acc.grid_code[3] : acc.grid_last[3],
                         acc.grid_code[0] != 0.0 ? acc.grid_code[0] : acc.grid_last[0],
                         acc.grid_code[1] != 0.0 ? acc.grid_code[1] : acc.grid_last[1]};
  const double scale[6] = {1.0, a.scale_obstacle, a.scale_goal_front, a.scale_alignment, a.scale_path, a.scale_goal};
  double total = 0.0;
  bool done = false;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double term = 0.0;  // what this critic adds; negative = rejecting code; skipped critics add nothing
    if (scale[k] != 0.0) {
      double cst = raw[k];
      if (cst < 0) term = cst;
      else {
        if (cst != 0) cst *= scale[k];
        term = cst;
      }
    }
    if (terms_out && lane == 0) terms_out[k] = scale[k] == 0.0 ? 0.0 : term;
    if (!done) {
      if (term < 0) {
        total = term;
        done = true;
      } else {
        total += term;
      }
    }
  }
  return total;
}

// OscillationCostFunction::scoreTrajectory (oscillation_cost_function.cpp:166-176) on the latched-flag mask
__device__ __forceinline__ bool oscillation_rejects(int m, double xv, double yv, double thv) {
  return ((m & 1) && xv < 0.0) || ((m & 2) && xv > 0.0) || ((m & 4) && yv < 0.0) || ((m & 8) && yv > 0.0) ||
         ((m & 16) && thv < 0.0) || ((m & 32) && thv > 0.0);
}

__device__ __forceinline__ float sample_vx(const DwaScoreArgs& a, int i) { return a.inline_samples ? a.samples_inline[i] : a.vxs[i]; }
__device__ __forceinline__ float sample_vy(const DwaScoreArgs& a, int i) { return a.inline_samples ? a.samples_inline[a.nx + i] : a.vys[i]; }
__device__ __forceinline__ float sample_vth(const DwaScoreArgs& a, int i) {
  return a.inline_samples ? a.samples_inline[a.nx + a.ny + i] : a.vths[i];
}

// scores one velocity sample with a whole warp; points_out (nullable) receives 3 doubles per trajectory point.
// kScore = false only generates the trajectory (points, step count): the critics are skipped and cost stays NaN.
constexpr int kWarpScratchDoubles = 128 + 16 + 16 * kMaxFootprint;  // 4 x 32 pose doubles, 32 ints, 32 x kMaxFootprint vertex cells
template <bool kScore>
__device__ TrajResult score_sample(const DwaScoreArgs& a, long long sample, int lane, double* terms_out,
                                   double* points_out, int points_capacity, double* warp_scratch,
                                   const uint8_t* __restrict__ cost) {
  TrajResult res;
  res.cost = nan_quiet();
  res.generated = false;
  res.num_steps = 0;
  const int ith = (int)(sample % a.nth);
  const long long t1 = sample / a.nth;
  const int iy = (int)(t1 % a.ny), ix = (int)(t1 / a.ny);
  const float svx = sample_vx(a, ix), svy = sample_vy(a, iy), svth = sample_vth(a, ith);

  // generateTrajectory :186-216
  const double vmag = hypot((double)svx, (double)svy);
  const double eps = 1e-4;
  if ((a.min_trans_vel >= 0 && vmag + eps < a.min_trans_vel) && (a.min_rot_vel >= 0 && fabs((double)svth) + eps < a.min_rot_vel))
    return res;
  if (a.max_trans_vel >= 0 && vmag - eps > a.max_trans_vel) return res;
  const double sim_time_distance = vmag * a.sim_time;
  const double sim_time_angle = fabs((double)svth) * a.sim_time;
  const int num_steps = (int)ceil(fmax(sim_time_distance / a.sim_granularity, sim_time_angle / a.angular_sim_granularity));
  if (num_steps <= 0) return res;
  const double dt = a.sim_time / num_steps;
  res.generated = true;
  res.num_steps = num_steps;

  const bool continued = !a.use_dwa;
  float lvx = svx, lvy = svy, lvth = svth;  // loop_vel
  auto new_vel = [&](float v, float target, float acc) -> float {  // computeNewVelocities :265-276
    if (v < target) return (float)fmin((double)target, v + acc * dt);
    return (float)fmax((double)target, v - acc * dt);
  };
  if (continued) {
    lvx = new_vel(a.vel[0], svx, a.acc[0]);
    lvy = new_vel(a.vel[1], svy, a.acc[1]);
    lvth = new_vel(a.vel[2], svth, a.acc[2]);
  }
  const float txv = lvx, tyv = lvy, tthv = lvth;  // traj.xv_, yv_, thetav_

  // OscillationCostFunction (scale 1): sign of the sampled velocity against the latched flags
  const double xv = txv, yv = tyv, thv = tthv;
  const bool osc_bad = oscillation_rejects(a.osc_mask, xv, yv, thv);

  float sx = a.pos[0], sy = a.pos[1], sth = a.pos[2];  // state at the first point of the current round
  CriticAcc acc;
  critic_acc_init(acc);

  for (int base = 0; base < num_steps; base += 32) {
    const int cnt = min(32, num_steps - base);
    // heading (and velocity) recurrence, replayed by every lane; lane l keeps the values of step base + l
    float th = sth, my_th = sth, my_vx = lvx, my_vy = lvy;
    for (int l = 0; l < cnt; ++l) {
      if (lane == l) my_th = th;
      if (continued) {
        lvx = new_vel(lvx, svx, a.acc[0]);
        lvy = new_vel(lvy, svy, a.acc[1]);
        lvth = new_vel(lvth, svth, a.acc[2]);
      }
      if (lane == l) { my_vx = lvx; my_vy = lvy; }
      th = (float)((double)th + lvth * dt);  // computeNewPositions :258
    }
    // trig of my own step, fp64 on the float heading (:256-257)
    const double thd = (double)my_th;
    double c, s;
    sincos(thd, &s, &c);
    double ddx = my_vx * c, ddy = my_vx * s;
    if (my_vy != 0.0f) {
      double c2, s2;  // cos / sin of the same argument: one range reduction
      sincos(M_PI_2 + thd, &s2, &c2);
      ddx = ddx + my_vy * c2;
      ddy = ddy + my_vy * s2;
    } else {
      ddx = ddx + 0.0;
      ddy = ddy + 0.0;
    }
    ddx = ddx * dt;
    ddy = ddy * dt;
    // x / y prefix in the reference's order: pos = float(pos + delta) per step
    // (the per-step deltas are broadcast through the warp's scratch: one 8-byte shared load instead of two shuffles)
    float x = sx, y = sy, my_x = sx, my_y = sy;
    warp_scratch[lane] = ddx;
    warp_scratch[32 + lane] = ddy;
    __syncwarp();
    for (int l = 0; l < cnt; ++l) {
      if (lane == l) { my_x = x; my_y = y; }
      const double dxl = warp_scratch[l], dyl = warp_scratch[32 + l];
      x = (float)((double)x + dxl);
      y = (float)((double)y + dyl);
    }
    __syncwarp();  // the scratch is rewritten below (and by the next round)
    sx = x;
    sy = y;
    sth = th;

    const bool active = lane < cnt;
    const double px = my_x, py = my_y;
    if (points_out && active && base + lane < points_capacity) {
      points_out[3 * (base + lane)] = px;
      points_out[3 * (base + lane) + 1] = py;
      points_out[3 * (base + lane) + 2] = thd;
    }
    if (!kScore) continue;
    score_round(a, cost, lane, cnt, px, py, c, s, warp_scratch, acc);
  }

  if (!kScore) return res;
  res.cost = combine_critics(a, osc_bad, acc, terms_out, lane);
  return res;
}

// Regenerates the winning trajectory (its points are what findBestTrajectory copies out, :123-134) with one warp;
// `cost` is the total the scoring pass found for it.  idx < 0: nothing valid (result_traj_.cost_ = -7,
// dwa_planner.cpp:316).
__device__ void finish_winner(const DwaScoreArgs& a, long long idx, double cost, DwaDeviceResult* out, double* points,
                              int points_capacity, double* warp_scratch, unsigned* n_generated) {
  const int lane = threadIdx.x & 31;
  TrajResult r;
  r.generated = false;
  r.num_steps = 0;
  if (idx >= 0) r = score_sample<false>(a, idx, lane, nullptr, points, points_capacity, warp_scratch, a.g.cost);
  if (lane == 0) {
    out->n_scored = (int)*n_generated;  // samples the generator accepted; re-armed for the next search
    *n_generated = 0;
    if (idx >= 0 && r.generated && cost >= 0) {
      const int ith = (int)(idx % a.nth);
      const long long t1 = idx / a.nth;
      const int iy = (int)(t1 % a.ny), ix = (int)(t1 / a.ny);
      float vx = sample_vx(a, ix), vy = sample_vy(a, iy), vth = sample_vth(a, ith);
      if (!a.use_dwa) {  // traj.xv_ is the first accelerated velocity (:221-227)
        const double dt = a.sim_time / r.num_steps;
        auto nv = [&](float v, float target, float acc) -> float {
          if (v < target) return (float)fmin((double)target, v + acc * dt);
          return (float)fmax((double)target, v - acc * dt);
        };
        vx = nv(a.vel[0], vx, a.acc[0]);
        vy = nv(a.vel[1], vy, a.acc[1]);
        vth = nv(a.vel[2], vth, a.acc[2]);
      }
      out->cost = cost;
      out->xv = vx;
      out->yv = vy;
      out->thetav = vth;
      out->best_index = idx;
      out->n_points = min(r.num_steps, points_capacity);
    } else {
      out->cost = -7.0;  // dwa_planner.cpp:316
      out->best_index = -1;
      out->n_points = -1;  // host keeps its stale velocities / points, like result_traj_ does
    }
  }
}

// lexicographic (cost, index) minimum: the reference keeps the FIRST sample with the strictly smallest cost
__device__ __forceinline__ bool better(double c1, long long i1, double c2, long long i2) {
  return c1 < c2 || (c1 == c2 && i1 < i2);
}

// The exchange step of a sharded sweep, run by warp 0 of the last CTA of every rank's k_dwa_score.  Lane r < world
// delivers this rank's record to rank r's buffer (a peer-mapped address: the store crosses NVLink), a system-wide fence
// orders it before the sequence number; then lane r waits for rank r's record of this sweep in the LOCAL buffer.  The
// winner is the reference's: smallest cost, lowest sample index on equal cost (simple_scored_sampling_planner.cpp:111-116
// keeps the first strictly smaller one), whatever the partition.  A peer that never answers (its process died) ends
// the wait after two seconds with "nothing valid" rather than hanging the GPU.
__device__ __noinline__ void shard_exchange(ShardExchange* peer_of_lane, ShardExchange* mine, int world, int me,
                                            unsigned long long seq, unsigned* counters, double* cost_io, long long* index_io) {
  const int lane = threadIdx.x & 31;
  const int parity = (int)(seq & 1ull);
  const unsigned generated = counters[1];
  const double cost = *cost_io;
  const long long index = *index_io;
  if (lane < world) {
    ShardSlot* out = &peer_of_lane->slot[parity][me];
    out->cost = cost;
    out->index = index;
    out->generated = generated;
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(&out->seq) = seq;
  }
  double c = INFINITY;
  long long ix = -1;
  unsigned gen = 0;
  if (lane < world) {
    const ShardSlot* in = &mine->slot[parity][lane];
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    bool arrived = true;
    while (*reinterpret_cast<const volatile unsigned long long*>(&in->seq) != seq) {
      unsigned long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 2000000000ull) {
        arrived = false;
        break;
      }
    }
    __threadfence_system();
    if (arrived) {
      c = *reinterpret_cast<const volatile double*>(&in->cost);
      ix = *reinterpret_cast<const volatile long long*>(&in->index);
      gen = *reinterpret_cast<const volatile unsigned*>(&in->generated);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double oc = __shfl_xor_sync(0xffffffffu, c, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, ix, o);
    gen += __shfl_xor_sync(0xffffffffu, gen, o);
    if (oi >= 0 && (ix < 0 || better(oc, oi, c, ix))) {
      c = oc;
      ix = oi;
    }
  }
  __syncwarp();
  if (lane == 0) {
    *cost_io = c;
    *index_io = ix;
    counters[1] = gen;  // n_scored of the whole sweep (finish_winner reports and clears it)
  }
  __syncwarp();
}

__global__ void __launch_bounds__(kDwaWarpsPerBlock * 32, 4) k_dwa_score(DwaScoreArgs a) {
  // (the 14.4 KB local costmap is read through L1: a per-CTA copy in shared memory measured 3-5 % slower)
  const uint8_t* costmap = a.g.cost;
  __shared__ double s_cost[kDwaWarpsPerBlock];
  __shared__ long long s_index[kDwaWarpsPerBlock];
  __shared__ int s_generated[kDwaWarpsPerBlock];
  __shared__ bool s_last;
  __shared__ double s_scratch[kDwaWarpsPerBlock][kWarpScratchDoubles];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long sample = a.begin + ((long long)blockIdx.x * a.stride_world + a.stride_rank) * kDwaWarpsPerBlock + warp;
  // Launched with programmatic stream serialization behind the MapGrid kernel, which runs on four SMs for tens of
  // microseconds: the rollout and the footprint walks (costmap only) start right away, and score_sample waits for the
  // distance grids (cudaGridDependencySynchronize) just before its first look-up.
  double cost = INFINITY;
  long long index = -1;
  int generated = 0;
  if (sample < a.end) {
    double* terms = a.all_terms ? a.all_terms + 6 * (sample - a.begin) : nullptr;
    const TrajResult r = score_sample<true>(a, sample, lane, terms, nullptr, 0, s_scratch[warp], costmap);
    generated = r.generated;
    if (terms && !r.generated && lane == 0)
      for (int k = 0; k < 6; ++k) terms[k] = nan_quiet();
    if (r.generated && r.cost >= 0) {
      cost = r.cost;
      index = sample;
    }
  }
  if (lane == 0) {
    s_cost[warp] = cost;
    s_index[warp] = index;
    s_generated[warp] = generated;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double bc = INFINITY;
    long long bi = -1;
    int gen = 0;
    for (int wdx = 0; wdx < kDwaWarpsPerBlock; ++wdx) {
      gen += s_generated[wdx];
      if (s_index[wdx] >= 0 && (bi < 0 || better(s_cost[wdx], s_index[wdx], bc, bi))) {
        bc = s_cost[wdx];
        bi = s_index[wdx];
      }
    }
    a.block_cost[blockIdx.x] = bc;
    a.block_index[blockIdx.x] = bi;
    if (gen) atomicAdd(&a.counters[1], (unsigned)gen);
    __threadfence();
    s_last = atomicAdd(&a.counters[0], 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  // the last CTA to finish reduces the per-CTA minima
  __threadfence();
  double bc = INFINITY;
  long long bi = -1;
  for (unsigned i = threadIdx.x; i < gridDim.x; i += blockDim.x) {
    const double c = a.block_cost[i];
    const long long ix = a.block_index[i];
    if (ix >= 0 && (bi < 0 || better(c, ix, bc, bi))) {
      bc = c;
      bi = ix;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double oc = __shfl_xor_sync(0xffffffffu, bc, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (oi >= 0 && (bi < 0 || better(oc, oi, bc, bi))) {
      bc = oc;
      bi = oi;
    }
  }
  if (lane == 0) {
    s_cost[warp] = bc;
    s_index[warp] = bi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    bc = INFINITY;
    bi = -1;
    for (int wdx = 0; wdx < kDwaWarpsPerBlock; ++wdx)
      if (s_index[wdx] >= 0 && (bi < 0 || better(s_cost[wdx], s_index[wdx], bc, bi))) {
        bc = s_cost[wdx];
        bi = s_index[wdx];
      }
    *a.best_cost = bc;
    *a.best_index = bi;
    a.counters[0] = 0;  // re-armed for the next launch (counters[1] is read and cleared by the finishing step)
    s_cost[0] = bc;
    s_index[0] = bi;
  }
  if (a.finish_out == nullptr) return;
  __syncthreads();
  if (warp != 0) return;
  if (a.shard_peer[0] != nullptr)  // multi-GPU sweep: the winner of all ranks
    shard_exchange(lane < a.stride_world ? a.shard_peer[lane] : nullptr, a.shard_peer[a.stride_rank], a.stride_world,
                   a.stride_rank, a.shard_seq, a.counters, &s_cost[0], &s_index[0]);
  finish_winner(a, s_index[0], s_cost[0], a.finish_out, a.finish_points, a.finish_capacity, s_scratch[0], &a.counters[1]);
}

// DWAPlanner::checkTrajectory: one warp scores sample 0 of a one-sample argument block; a rejected sample leaves an
// empty trajectory, which every critic scores as 0 (an empty footprint still answers -9)
__global__ void k_dwa_check(DwaScoreArgs a, double* cost_out) {
  __shared__ double s_scratch[kWarpScratchDoubles];
  const TrajResult r = score_sample<true>(a, 0, threadIdx.x & 31, nullptr, nullptr, 0, s_scratch, a.g.cost);
  if (threadIdx.x == 0) *cost_out = r.generated ? r.cost : ((a.nfp == 0 && a.scale_obstacle != 0.0) ? -9.0 : 0.0);
}

// The batched base_local_planner::TrajectoryCostFunction backend (trajectory_cost_function.h:52-82): trajectories the
// CALLER generated (any TrajectorySampleGenerator) are scored by the six critics DWAPlanner wires up, in its order
// (dwa_planner.cpp:167-173), with SimpleScoredSamplingPlanner::scoreTrajectory's accumulation (:50-79, no early exit).
// One warp per trajectory, one lane per point of a round; points = x, y, theta as Trajectory::getPoint returns them
// (doubles), vels = xv_, yv_, thetav_.  A trajectory without points scores what the reference's critics return for
// an empty loop: 0 from every grid / obstacle critic (-9 for an empty footprint), -5 from a latched oscillation flag.
__global__ void __launch_bounds__(kDwaWarpsPerBlock * 32) k_dwa_score_points(DwaScoreArgs a, const int* __restrict__ offsets,
                                                                           const double* __restrict__ points,
                                                                           const double* __restrict__ vels, int n_traj,
                                                                           double* __restrict__ costs_out,
                                                                           double* __restrict__ terms_out) {
  __shared__ double s_scratch[kDwaWarpsPerBlock][kWarpScratchDoubles];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int t = blockIdx.x * kDwaWarpsPerBlock + warp;
  if (t >= n_traj) return;
  const int first = offsets[t], n = offsets[t + 1] - first;
  const bool osc_bad = oscillation_rejects(a.osc_mask, vels[3 * t], vels[3 * t + 1], vels[3 * t + 2]);
  CriticAcc acc;
  critic_acc_init(acc);
  for (int base = 0; base < n; base += 32) {
    const int cnt = min(32, n - base);
    double px = 0.0, py = 0.0, c = 1.0, s = 0.0;
    if (lane < cnt) {
      const double* p = points + 3 * (size_t)(first + base + lane);
      px = p[0];
      py = p[1];
      sincos(p[2], &s, &c);  // WorldModel::footprintCost / MapGridCostFunction take cos, sin of the point's heading
    }
    score_round(a, a.g.cost, lane, cnt, px, py, c, s, s_scratch[warp], acc);
    __syncwarp();
  }
  const double total = combine_critics(a, osc_bad, acc, terms_out ? terms_out + 6 * (size_t)t : nullptr, lane);
  if (lane == 0) costs_out[t] = total;
}

// stand-alone finish for sharded sweeps: the winner was chosen from the all-gathered per-rank minima
__global__ void k_dwa_finish(DwaScoreArgs a, long long forced_index, double forced_cost, DwaDeviceResult* out,
                             double* points, int points_capacity) {
  __shared__ double s_scratch[kWarpScratchDoubles];
  finish_winner(a, forced_index, forced_cost, out, points, points_capacity, s_scratch, &a.counters[1]);
}

// all_explored costs exactly as the sequential search reports them (simple_scored_sampling_planner.cpp:50-79,
// 99-110): a sample's critic sum stops at the first critic after which it exceeds the best cost found BEFORE it.
// One CTA walks the samples in order carrying that running best.
__global__ void k_dwa_report(const double* __restrict__ terms, double* __restrict__ reported, long long n) {
  __shared__ double s_full[1024];
  __shared__ double s_prefix[1024];
  __shared__ double s_carry;
  if (threadIdx.x == 0) s_carry = -1.0;  // best_traj_cost = -1
  __syncthreads();
  for (long long base = 0; base < n; base += blockDim.x) {
    const long long i = base + threadIdx.x;
    double t[6];
    double full = nan_quiet();
    bool gen = false;
    if (i < n) {
      for (int k = 0; k < 6; ++k) t[k] = terms[6 * i + k];
      gen = !isnan(t[0]);
      if (gen) {
        full = 0.0;
        for (int k = 0; k < 6; ++k) {
          if (t[k] < 0) { full = t[k]; break; }
          full += t[k];
        }
      }
    }
    s_full[threadIdx.x] = (gen && full >= 0) ? full : INFINITY;
    __syncthreads();
    if (threadIdx.x == 0) {  // exclusive running minimum over this chunk, seeded with the carry
      double best = s_carry;
      for (int j = 0; j < (int)blockDim.x; ++j) {
        s_prefix[j] = best;
        const double f = s_full[j];
        if (f != INFINITY && (best < 0 || f < best)) best = f;
      }
      s_carry = best;
    }
    __syncthreads();
    if (i < n) {
      double rep = nan_quiet();
      if (gen) {
        const double best = s_prefix[threadIdx.x];
        rep = 0.0;
        for (int k = 0; k < 6; ++k) {
          // a critic with scale 0 is skipped before the early-exit test: its stored term is exactly 0 and the
          // running sum cannot newly exceed best, so testing after it is equivalent
          if (t[k] < 0) { rep = t[k]; break; }
          rep += t[k];
          if (best > 0 && rep > best) break;
        }
      }
      reported[i] = rep;
    }
    __syncthreads();
  }
}


// ---------------------------------------------------------------------------------------------------------------
// Fleet mode (config C5): many independent robots, each with its own local costmap, plan, pose, velocity and
// oscillation mask, scored in ONE launch.  A CTA serves one robot: it copies the shared DwaScoreArgs into shared
// memory, patches the robot's fields in, and runs the very same score_sample as the single-planner kernel.
__device__ __forceinline__ void fleet_patch_args(DwaScoreArgs& s_a, const DwaScoreArgs& base, const FleetRobot& r,
                                                 const float* samples) {
  // cooperative word copy of the shared arguments, then the robot's own fields
  const uint32_t* src = reinterpret_cast<const uint32_t*>(&base);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&s_a);
  constexpr int kHeadWords = (int)(offsetof(DwaScoreArgs, samples_inline) / 4);
  constexpr int kTailStart = (int)((offsetof(DwaScoreArgs, samples_inline) + sizeof(float) * kInlineSamples) / 4);
  constexpr int kWords = (int)(sizeof(DwaScoreArgs) / 4);
  for (int i = threadIdx.x; i < kHeadWords; i += blockDim.x) dst[i] = src[i];
  for (int i = kTailStart + threadIdx.x; i < kWords; i += blockDim.x) dst[i] = src[i];
  const int n_s = r.nx + r.ny + r.nth;
  for (int i = threadIdx.x; i < n_s; i += blockDim.x) s_a.samples_inline[i] = samples[r.samples_offset + i];
  __syncthreads();
  if (threadIdx.x == 0) {
    s_a.g = r.grids.g;
    for (int k = 0; k < 4; ++k) s_a.dist[k] = r.grids.job[k].dist;
    s_a.nx = r.nx; s_a.ny = r.ny; s_a.nth = r.nth;
    s_a.inline_samples = 1;
    for (int k = 0; k < 3; ++k) { s_a.pos[k] = r.pos[k]; s_a.vel[k] = r.vel[k]; }
    s_a.osc_mask = r.osc_mask;
    s_a.scale_alignment = r.scale_alignment;
    s_a.begin = 0;
    s_a.end = (long long)r.nx * r.ny * r.nth;
    s_a.all_terms = nullptr;
    s_a.finish_out = nullptr;
  }
  __syncthreads();
}

// grid = n_robots * blocks_per_robot CTAs; per CTA the (cost, index) minimum of its 8 samples
__global__ void __launch_bounds__(kDwaWarpsPerBlock * 32, 4) k_fleet_score(DwaScoreArgs base, const FleetRobot* robots,
                                                                        const float* samples, int blocks_per_robot,
                                                                        double* block_cost, long long* block_index,
                                                                        unsigned* generated) {
  __shared__ DwaScoreArgs s_a;
  __shared__ double s_cost[kDwaWarpsPerBlock];
  __shared__ long long s_index[kDwaWarpsPerBlock];
  __shared__ int s_generated[kDwaWarpsPerBlock];
  __shared__ double s_scratch[kDwaWarpsPerBlock][kWarpScratchDoubles];
  const int robot = blockIdx.x / blocks_per_robot, local = blockIdx.x % blocks_per_robot;
  const FleetRobot& r = robots[robot];
  if ((long long)local * kDwaWarpsPerBlock >= (long long)r.nx * r.ny * r.nth) {  // no samples for this CTA
    if (threadIdx.x == 0) {
      block_cost[blockIdx.x] = INFINITY;
      block_index[blockIdx.x] = -1;
    }
    return;
  }
  fleet_patch_args(s_a, base, r, samples);
  const uint8_t* costmap = s_a.g.cost;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long sample = (long long)local * kDwaWarpsPerBlock + warp;
  double cost = INFINITY;
  long long index = -1;
  int gen = 0;
  if (sample < s_a.end) {
    const TrajResult t = score_sample<true>(s_a, sample, lane, nullptr, nullptr, 0, s_scratch[warp], costmap);
    gen = t.generated;
    if (t.generated && t.cost >= 0) {
      cost = t.cost;
      index = sample;
    }
  }
  if (lane == 0) {
    s_cost[warp] = cost;
    s_index[warp] = index;
    s_generated[warp] = gen;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double bc = INFINITY;
    long long bi = -1;
    int g = 0;
    for (int wdx = 0; wdx < kDwaWarpsPerBlock; ++wdx) {
      g += s_generated[wdx];
      if (s_index[wdx] >= 0 && (bi < 0 || better(s_cost[wdx], s_index[wdx], bc, bi))) {
        bc = s_cost[wdx];
        bi = s_index[wdx];
      }
    }
    block_cost[blockIdx.x] = bc;
    block_index[blockIdx.x] = bi;
    if (g) atomicAdd(&generated[robot], (unsigned)g);
  }
}

// raw local maps [n][sy][sx] (contiguous) -> the stacked, padded layer grid: robot r's row y lands on row
// r * stride + y with row pitch `pitch`; pad rows and pad columns are never written (they stay zero)
__global__ void k_fleet_scatter_maps(const uint8_t* __restrict__ raw, uint8_t* __restrict__ stacked, unsigned sx,
                                     unsigned sy, unsigned stride, unsigned pitch, unsigned n) {
  const size_t row = (size_t)blockIdx.x * blockDim.y + threadIdx.y;  // row over all robots
  if (row >= (size_t)n * sy) return;
  const unsigned r = (unsigned)(row / sy), y = (unsigned)(row - (size_t)r * sy);
  const uint8_t* src = raw + row * sx;
  uint8_t* dst = stacked + ((size_t)r * stride + y) * pitch;
  if ((sx & 3u) == 0 && (((size_t)src) & 3u) == 0) {
    for (unsigned x = threadIdx.x * 4; x < sx; x += blockDim.x * 4)
      *reinterpret_cast<uint32_t*>(dst + x) = *reinterpret_cast<const uint32_t*>(src + x);
  } else {
    for (unsigned x = threadIdx.x; x < sx; x += blockDim.x) dst[x] = src[x];
  }
}

// one warp (= one CTA) per robot: reduce its CTAs' minima with the first-strictly-smaller rule and fill the result
__global__ void __launch_bounds__(32) k_fleet_finish(DwaScoreArgs base, const FleetRobot* robots, const float* samples,
                                                     int blocks_per_robot, const double* block_cost,
                                                     const long long* block_index, unsigned* generated,
                                                     DwaDeviceResult* results) {
  __shared__ DwaScoreArgs s_a;
  __shared__ double s_scratch[kWarpScratchDoubles];
  const int robot = blockIdx.x, lane = threadIdx.x;
  fleet_patch_args(s_a, base, robots[robot], samples);
  double bc = INFINITY;
  long long bi = -1;
  for (int i = lane; i < blocks_per_robot; i += 32) {
    const double c = block_cost[(size_t)robot * blocks_per_robot + i];
    const long long ix = block_index[(size_t)robot * blocks_per_robot + i];
    if (ix >= 0 && (bi < 0 || better(c, ix, bc, bi))) {
      bc = c;
      bi = ix;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double oc = __shfl_xor_sync(0xffffffffu, bc, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (oi >= 0 && (bi < 0 || better(oc, oi, bc, bi))) {
      bc = oc;
      bi = oi;
    }
  }
  finish_winner(s_a, bi, bc, results + robot, nullptr, 0, s_scratch, generated + robot);
}

// DWAPlanner::checkTrajectory of any robots' candidates in one launch (navgpu_fleet_check_trajectories): one warp (= one
// CTA) per candidate.  Each robot's record is a one-sample block (nx = ny = nth = 1, samples_offset 0), so passing the
// candidate's own 3 floats as the sample array makes it sample 0 -- k_dwa_check's way, with its cost rule.  (A minimum
// of one CTA per SM lets ptxas keep the values live across the sincos slow path in registers instead of spilling them.)
__global__ void __launch_bounds__(32, 1) k_fleet_check(DwaScoreArgs base, const FleetRobot* robots,
                                                    const int* __restrict__ robot_of, const float* __restrict__ candidates,
                                                    double* __restrict__ costs) {
  __shared__ DwaScoreArgs s_a;
  __shared__ double s_scratch[kWarpScratchDoubles];
  const int c = blockIdx.x;
  fleet_patch_args(s_a, base, robots[robot_of[c]], candidates + 3 * (size_t)c);
  const TrajResult r = score_sample<true>(s_a, 0, threadIdx.x & 31, nullptr, nullptr, 0, s_scratch, s_a.g.cost);
  if (threadIdx.x == 0) costs[c] = r.generated ? r.cost : ((s_a.nfp == 0 && s_a.scale_obstacle != 0.0) ? -9.0 : 0.0);
}

// ---------------------------------------------------------------------------------------------------------------
// The device fleet step (navgpu_fleet_step_device): what navgpu_fleet_step does per robot on the host, one thread per
// robot, with the host step's own functions (fleet_roll_step, enumerate_samples, Oscillation, apply_dwa_result).
constexpr int kFleetRobotThreads = 128;
constexpr uint8_t kFleetActive = 1, kFleetAligned = 2;  // per-robot flags: planned by the steps; alignment grid = path grid

struct FleetPrepareArgs {
  const double* poses;  // [n][3], device memory
  const double* vels;
  FleetRobot* robots;
  FleetDwaState* state;
  const uint8_t* flags;
  float* samples;  // robot r's per-axis samples at r * slot
  int slot, n;
  navgpu_dwa_config cfg;
  FleetCmStep* steps;  // sensing fleets: the costmap update's step records; null on raw-map fleets
  unsigned sx, sy;
  double res;
};

// Before the costmap update: a sensing fleet's roll of every robot (fleet_costmap_roll), whose origin also goes into
// the robot's MapGrid record; then, for robots the steps plan, the record's per-step fields and velocity samples
// (navgpu_fleet_step's per-robot loop).  A left-out robot gets no samples, so its scoring CTAs exit at once.
__global__ void __launch_bounds__(kFleetRobotThreads) k_fleet_prepare(FleetPrepareArgs a) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= a.n) return;
  const double pose[3] = {a.poses[3 * r], a.poses[3 * r + 1], a.poses[3 * r + 2]};
  FleetRobot& R = a.robots[r];
  FleetDwaState& S = a.state[r];
  if (a.steps) {
    const FleetCmStep st = fleet_roll_step(pose, S.origin[0], S.origin[1], a.sx, a.sy, a.res);
    a.steps[r] = st;
    S.origin[0] = st.ox;
    S.origin[1] = st.oy;
    R.grids.g.ox = st.ox;
    R.grids.g.oy = st.oy;
  }
  R.samples_offset = r * a.slot;
  if (!(a.flags[r] & kFleetActive)) {
    R.nx = R.ny = R.nth = 0;
    return;
  }
  const float pos[3] = {(float)pose[0], (float)pose[1], (float)pose[2]};
  const float vel[3] = {(float)a.vels[3 * r], (float)a.vels[3 * r + 1], (float)a.vels[3 * r + 2]};
  const float goal[2] = {0.f, 0.f};  // (use_dwa = 0 only, which device steps refuse)
  int counts[3];
  enumerate_samples(a.cfg, pos, vel, goal, a.samples + (size_t)r * a.slot, counts);
  for (int k = 0; k < 3; ++k) { R.pos[k] = pos[k]; R.vel[k] = vel[k]; }
  R.osc_mask = S.osc.mask();
  R.nx = counts[0]; R.ny = counts[1]; R.nth = counts[2];
}

// After k_fleet_finish: the host step's epilogue per planned robot (apply_dwa_result: result_traj_'s velocities, the
// oscillation flags, the result record), the record written to the caller's device buffer; left-out robots' records
// and state stay as they are
__global__ void __launch_bounds__(kFleetRobotThreads) k_fleet_apply(navgpu_dwa_config cfg, const double* poses,
                                                                    const FleetRobot* robots, const uint8_t* flags,
                                                                    const DwaDeviceResult* found, FleetDwaState* state,
                                                                    navgpu_dwa_result* results, int n) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n || !(flags[r] & kFleetActive)) return;
  const FleetRobot& R = robots[r];
  FleetDwaState S = state[r];
  navgpu_dwa_result out;
  apply_dwa_result(found[r], cfg, poses + 3 * r, R.nx * R.ny * R.nth, S.res_v, S.osc, &out);
  out.n_points = 0;
  S.planned = 1;
  S.aliased = (flags[r] & kFleetAligned) ? 1 : 0;
  state[r] = S;
  results[r] = out;
}

}  // namespace navgpu
