// mirror_kernels.cuh -- keeping a HOST copy of the master grid in sync without shipping the whole grid every cycle.
//
// The reference's consumers (Costmap2DROS, the planners, Costmap2DPublisher) read the master Costmap2D in host memory
// after LayeredCostmap::updateMap (layered_costmap.cpp:79-150).  A device-resident master grid therefore has to reach the
// host every cycle, and at 4000 x 4000 that copy (16 MB over PCIe, ~0.3 ms) costs four times the update itself --
// although all but a few hundred cells keep their value from one cycle to the next.  The device keeps a SHADOW of what
// the host mirror holds; k_mirror_diff compares the master grid with it tile by tile, writes the tiles that differ
// straight into mapped pinned host memory (posted writes over PCIe) and brings the shadow up to date: into their own
// place in the host mirror when that buffer is page-locked (navgpu_host_register), else compacted into a staging area
// from which the call scatters them.  Either way the mirror is byte-identical to the master grid again, whatever
// happened in between (skipped cycles, rolled origins, navgpu_costmap_set).
#pragma once

#include "common.cuh"

namespace navgpu {

constexpr int kMirrorTileW = 128, kMirrorTileH = 16;            // one warp per tile: 8 lanes x 16 B per row, 4 rows per pass
constexpr int kMirrorTileBytes = kMirrorTileW * kMirrorTileH;  // 2 KB
constexpr int kMirrorWarps = 8;

struct MirrorCtl {  // mapped pinned host memory: written by the last CTA of k_mirror_diff
  unsigned n_changed;  // tiles that differ (may exceed the staging capacity: then the host copies the whole grid)
  unsigned n_staged;   // tiles actually written to the staging buffer = min(n_changed, capacity)
  DevWindow win;       // the window of the last update cycle, so that one synchronisation serves both
  // written last, behind a system-scope fence: the call's number.  The host polls this word instead of synchronising the
  // stream (the documented mapped-memory signalling pattern: data, __threadfence_system(), flag), which takes the
  // stream-synchronisation wake-up out of every cycle.
  unsigned seq;
};

struct MirrorArgs {
  const uint8_t* master;
  uint8_t* shadow;
  unsigned sx, sy, pitch;
  unsigned tiles_x, tiles_y;
  unsigned capacity;     // tiles the staging buffer holds
  uint8_t* stage;        // mapped pinned: capacity x kMirrorTileBytes
  unsigned* stage_tile;  // mapped pinned: tile number of every staged tile
  unsigned* counters;    // device: [0] changed tiles, [1] CTAs done
  MirrorCtl* ctl;        // mapped pinned
  const DevWindow* win;  // nullable
  // Where the master grid can differ from the shadow: the box the update cycles accumulated on the device since the
  // last call (finalize_bounds: every window grown by 2R), cut down to `hx0..hyn` when the host knows better (cycles that
  // recomputed the whole map from layers that only changed inside the obstacle kernels' boxes), or everything when
  // `all` is set (first call, uploads, rolled origins).  The last CTA empties the device box.
  DevWindow* dirty;
  int all;
  int hx0, hxn, hy0, hyn;
  // the grid covers the tiles [tx0, tx0 + tw) x [ty0, ty0 + th) only (all of them unless the host's box is smaller)
  unsigned tx0, ty0, tw, th;
  // non-null: the host mirror itself is page-locked and mapped (its address as this device sees it, rows host_pitch
  // bytes apart) -- changed tiles are written straight to their place in it and only their numbers are staged
  uint8_t* host_direct;
  unsigned host_pitch;
  unsigned seq;  // MirrorCtl::seq of this call
  // non-null: the sweep in front of this kernel was a whole-map cycle whose k_inflate publishes `inflate_epoch` per
  // 128 x 64 tile (inflate_pitch tiles per row) when the tile's cells are final: a tile is compared as soon as the
  // inflate tile that writes it is done, while the rest of that kernel is still running
  const unsigned* inflate_done = nullptr;
  unsigned inflate_epoch = 0;
  int inflate_pitch = 0;
};
constexpr int kMirrorInflateTileW = 128, kMirrorInflateTileH = 64;  // = k_inflate's tile (static_assert in costmap.cu)
static_assert(kMirrorTileW % kMirrorInflateTileW == 0 && kMirrorInflateTileH % kMirrorTileH == 0,
              "a mirror tile lies inside one row of inflate tiles");

__device__ __forceinline__ void mirror_wait_word(const unsigned* p, unsigned want) {
  unsigned seen;
  for (;;) {
    asm volatile("ld.acquire.gpu.u32 %0, [%1];" : "=r"(seen) : "l"(p) : "memory");
    if (seen == want) break;
    __nanosleep(100);
  }
}

// bytes of a and b that differ among the first n_valid bytes of the 16-byte group
__device__ __forceinline__ bool group_differs(const uint4& a, const uint4& b, int n_valid) {
  if (n_valid >= 16) return ((a.x ^ b.x) | (a.y ^ b.y) | (a.z ^ b.z) | (a.w ^ b.w)) != 0;
  const uint32_t d[4] = {a.x ^ b.x, a.y ^ b.y, a.z ^ b.z, a.w ^ b.w};
  uint32_t any = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int nb = min(4, max(0, n_valid - 4 * k));
    const uint32_t mask = nb >= 4 ? 0xffffffffu : ((1u << (8 * nb)) - 1u);
    any |= d[k] & mask;
  }
  return any != 0;
}

__global__ void __launch_bounds__(kMirrorWarps * 32) k_mirror_diff(MirrorArgs a) {
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // launched with programmatic stream serialization behind the cycle's last kernel: resident while that kernel drains,
  // reading nothing before it has completed
  if (a.inflate_done) {
    // Every CTA of the k_inflate grid in front is resident or done by now (it triggers the programmatic launch at its
    // first instruction).  Its tile (0, 0) depends on k_merge_seed's tile (0, 0), which waits for the END of the
    // obstacle kernel: behind this word the cycle's window and the dirty box are final.
    if (lane == 0) mirror_wait_word(a.inflate_done, a.inflate_epoch);
    __syncwarp();
  } else {
    cudaGridDependencySynchronize();
  }
  const unsigned local = blockIdx.x * kMirrorWarps + warp;  // index within the launched rectangle of tiles
  const unsigned n_tiles = a.tiles_x * a.tiles_y;
  const unsigned tile = local < a.tw * a.th ? (a.ty0 + local / a.tw) * a.tiles_x + a.tx0 + local % a.tw : n_tiles;
  int rx0 = 0, rxn = (int)a.sx, ry0 = 0, ryn = (int)a.sy;
  if (!a.all) {
    const DevWindow d = *a.dirty;  // (read by every CTA before the last one resets it: the reset follows the ticket)
    if (d.valid) {
      rx0 = max(d.x0, a.hx0); rxn = min(d.xn, a.hxn); ry0 = max(d.y0, a.hy0); ryn = min(d.yn, a.hyn);
    } else {
      rxn = ryn = 0;  // no update cycle since the last call
    }
  }
  const unsigned tx_ = tile % a.tiles_x, ty_ = tile / a.tiles_x;
  const bool in_region = (int)(tx_ * kMirrorTileW) < rxn && (int)((tx_ + 1) * kMirrorTileW) > rx0 &&
                         (int)(ty_ * kMirrorTileH) < ryn && (int)((ty_ + 1) * kMirrorTileH) > ry0;
  if (tile < n_tiles && in_region) {
    const unsigned tx = tx_, ty = ty_;
    if (a.inflate_done) {  // the inflate tile that covers this 128 x 16 tile
      if (lane < kMirrorTileW / kMirrorInflateTileW) {
        const int ix = (int)(tx * kMirrorTileW) / kMirrorInflateTileW + lane, iy = (int)(ty * kMirrorTileH) / kMirrorInflateTileH;
        if (ix < a.inflate_pitch) mirror_wait_word(a.inflate_done + iy * a.inflate_pitch + ix, a.inflate_epoch);
      }
      __syncwarp();
    }
    const int x = (int)tx * kMirrorTileW + (lane & 7) * 16;
    const int y0 = (int)ty * kMirrorTileH + (lane >> 3);
    const int n_valid = min(16, max(0, (int)a.sx - x));  // the row padding is nobody's data
    uint4 m[4], s[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int y = y0 + 4 * p;
      m[p] = s[p] = make_uint4(0, 0, 0, 0);
      if (y < (int)a.sy && n_valid > 0) {
        const size_t off = (size_t)y * a.pitch + x;
        m[p] = *reinterpret_cast<const uint4*>(a.master + off);
        s[p] = *reinterpret_cast<const uint4*>(a.shadow + off);
      }
    }
    bool differs = false;
#pragma unroll
    for (int p = 0; p < 4; ++p) differs |= group_differs(m[p], s[p], n_valid);
    if (__any_sync(0xffffffffu, differs)) {
      unsigned slot = 0;
      if (lane == 0) slot = atomicAdd(&a.counters[0], 1u);
      slot = __shfl_sync(0xffffffffu, slot, 0);
      const bool staged = slot < a.capacity;
      if (staged && lane == 0) a.stage_tile[slot] = tile;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int y = y0 + 4 * p;
        const bool in_map = y < (int)a.sy && n_valid > 0;
        if (a.host_direct) {
          if (in_map) {
            uint8_t* dst = a.host_direct + (size_t)y * a.host_pitch + x;
            if (n_valid == 16 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
              *reinterpret_cast<uint4*>(dst) = m[p];
            } else {
              const uint32_t w4[4] = {m[p].x, m[p].y, m[p].z, m[p].w};
              for (int b = 0; b < n_valid; ++b) dst[b] = (uint8_t)(w4[b >> 2] >> (8 * (b & 3)));
            }
          }
        } else if (staged) {  // rows below the map / columns right of it travel as zeros and are dropped by the host
          *reinterpret_cast<uint4*>(a.stage + (size_t)slot * kMirrorTileBytes + ((lane >> 3) + 4 * p) * kMirrorTileW +
                                    (lane & 7) * 16) = m[p];
        }
        if (in_map) *reinterpret_cast<uint4*>(a.shadow + (size_t)y * a.pitch + x) = m[p];
      }
    }
  }
  // the CTA that finishes last publishes the counts (and the cycle's window) and re-arms the counters
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();  // (this CTA's tiles are in host memory before its ticket counts)
    s_last = atomicAdd(&a.counters[1], 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last || threadIdx.x != 0) return;
  __threadfence_system();
  const unsigned n = *reinterpret_cast<volatile unsigned*>(&a.counters[0]);
  a.ctl->n_changed = n;
  a.ctl->n_staged = min(n, a.capacity);
  if (a.win) a.ctl->win = *a.win;
  a.counters[0] = 0;
  a.counters[1] = 0;
  a.dirty->valid = 0;
  __threadfence_system();
  *reinterpret_cast<volatile unsigned*>(&a.ctl->seq) = a.seq;
}

}  // namespace navgpu
