// ref_harness.cpp -- glue that exposes the reference's OWN compiled hot-path code through oracle_api.h.
//
// TEST INFRASTRUCTURE ONLY.  Compiled by oracle/Makefile together with the unmodified reference sources
// (read in place from /root/reference, never copied) into oracle/_ref/libnavref.so.
//
// What is reference code and what is restated here (because the enclosing reference TU needs ROS/PCL/tf):
//   reference, unmodified: Costmap2D, Layer, LayeredCostmap, CostmapLayer (all four updateWith*),
//       InflationLayer, raytraceLine/bresenham2D/MarkCell, setConvexPolygonCost, MapGrid, MapGridCostFunction,
//       ObstacleCostFunction, CostmapModel, LineIterator, OscillationCostFunction, SimpleTrajectoryGenerator,
//       VelocityIterator, SimpleScoredSamplingPlanner, Trajectory, calculateMinAndMaxDistances (via LayeredCostmap),
//       voxel_grid::VoxelGrid (markVoxelInMap, clearVoxelLineInMap = raytraceLine/bresenham3D/ClearVoxelInMap).
//   restated in this file: ObstacleLayer::updateBounds/raytraceFreespace/updateRaytraceBounds/updateFootprint/
//       updateCosts bodies (costmap_2d/plugins/obstacle_layer.cpp:340-448,498-610) on top of the reference's
//       protected CostmapLayer primitives; VoxelLayer::updateBounds/raytraceFreespace/updateOrigin/matchSize/resetMaps
//       (costmap_2d/plugins/voxel_layer.cpp:84-101,116-177,262-350,371-438) on top of the reference's VoxelGrid; StaticLayer::updateBounds/updateCosts non-rolling branch and
//       interpretValue (static_layer.cpp:149-163,263-299); transformFootprint and calculateMinAndMaxDistances
//       (footprint.cpp:41-67,106-120, that TU needs boost tokenizer + XmlRpc); DWAPlanner's wiring
//       (dwa_planner.cpp:52-112,116-182,240-286,292-319,357).
#include <costmap_2d/costmap_2d.h>
#include <costmap_2d/layered_costmap.h>
#include <costmap_2d/costmap_layer.h>
#include <costmap_2d/inflation_layer.h>
#include <costmap_2d/cost_values.h>
#include <costmap_2d/costmap_math.h>
#include <costmap_2d/observation.h>
#include <voxel_grid/voxel_grid.h>
#include <base_local_planner/map_grid.h>
#include <base_local_planner/map_grid_cost_function.h>
#include <base_local_planner/obstacle_cost_function.h>
#include <base_local_planner/oscillation_cost_function.h>
#include <base_local_planner/simple_trajectory_generator.h>
#include <base_local_planner/simple_scored_sampling_planner.h>
#include <base_local_planner/velocity_iterator.h>
#include <base_local_planner/line_iterator.h>
#include <base_local_planner/local_planner_limits.h>
#include <base_local_planner/costmap_model.h>
// the harness reads TrajectoryPlanner's private distance maps and oscillation flags (the reference translation unit
// itself is compiled untouched; access specifiers do not change the layout)
#define private public
#include <base_local_planner/trajectory_planner.h>
#undef private

#include <cmath>
#include <cstdio>
#include <limits>
#include <memory>
#include <queue>
#include <string>
#include <vector>

#include "oracle_api.h"
#include "scan_ingest_restated.h"
#include "plan_restated.h"

// ---- footprint.cpp needs boost::tokenizer/XmlRpc; its two pure functions are restated (footprint.cpp:41-67,106-120)
namespace costmap_2d {
void calculateMinAndMaxDistances(const std::vector<geometry_msgs::Point>& footprint, double& min_dist,
                                 double& max_dist) {
  min_dist = std::numeric_limits<double>::max();
  max_dist = 0.0;
  if (footprint.size() <= 2) return;
  for (unsigned int i = 0; i < footprint.size() - 1; ++i) {
    double vertex_dist = distance(0.0, 0.0, footprint[i].x, footprint[i].y);
    double edge_dist = distanceToLine(0.0, 0.0, footprint[i].x, footprint[i].y, footprint[i + 1].x, footprint[i + 1].y);
    min_dist = std::min(min_dist, std::min(vertex_dist, edge_dist));
    max_dist = std::max(max_dist, std::max(vertex_dist, edge_dist));
  }
  double vertex_dist = distance(0.0, 0.0, footprint.back().x, footprint.back().y);
  double edge_dist =
      distanceToLine(0.0, 0.0, footprint.back().x, footprint.back().y, footprint.front().x, footprint.front().y);
  min_dist = std::min(min_dist, std::min(vertex_dist, edge_dist));
  max_dist = std::max(max_dist, std::max(vertex_dist, edge_dist));
}

void transformFootprint(double x, double y, double theta, const std::vector<geometry_msgs::Point>& footprint_spec,
                        std::vector<geometry_msgs::Point>& oriented_footprint) {
  oriented_footprint.clear();
  double cos_th = cos(theta);
  double sin_th = sin(theta);
  for (unsigned int i = 0; i < footprint_spec.size(); ++i) {
    geometry_msgs::Point new_pt;
    new_pt.x = x + (footprint_spec[i].x * cos_th - footprint_spec[i].y * sin_th);
    new_pt.y = y + (footprint_spec[i].x * sin_th + footprint_spec[i].y * cos_th);
    oriented_footprint.push_back(new_pt);
  }
}
}  // namespace costmap_2d

namespace {

using costmap_2d::Costmap2D;
using costmap_2d::CostmapLayer;
using costmap_2d::LayeredCostmap;

// A CostmapLayer whose cells are supplied by the caller; merge policy selectable.  With TRUE_OVERWRITE / MAX it is
// StaticLayer's non-rolling behaviour (static_layer.cpp:263-299).
class GridLayer : public CostmapLayer {
 public:
  explicit GridLayer(int policy) : policy_(policy), x_(0), y_(0), width_(0), height_(0), has_updated_data_(false) {}
  void onInitialize() override {
    current_ = true;
    enabled_ = true;
    default_value_ = layered_costmap_->isTrackingUnknown() ? costmap_2d::NO_INFORMATION : costmap_2d::FREE_SPACE;
    matchSize();
  }
  void setData(const uint8_t* data) {
    memcpy(costmap_, data, size_t(size_x_) * size_y_);
    x_ = y_ = 0;
    width_ = size_x_;
    height_ = size_y_;
    has_updated_data_ = true;
  }
  void touchRegion(unsigned x, unsigned y, unsigned w, unsigned h) {
    x_ = x; y_ = y; width_ = w; height_ = h;
    has_updated_data_ = true;
  }
  void setEnabled(bool e) { enabled_ = e; }
  void updateBounds(double, double, double, double* min_x, double* min_y, double* max_x, double* max_y) override {
    if (!layered_costmap_->isRolling()) {
      if (!(has_updated_data_ || has_extra_bounds_)) return;
    }
    useExtraBounds(min_x, min_y, max_x, max_y);
    double wx, wy;
    mapToWorld(x_, y_, wx, wy);
    *min_x = std::min(wx, *min_x);
    *min_y = std::min(wy, *min_y);
    mapToWorld(x_ + width_, y_ + height_, wx, wy);
    *max_x = std::max(wx, *max_x);
    *max_y = std::max(wy, *max_y);
    has_updated_data_ = false;
  }
  void updateCosts(Costmap2D& master, int min_i, int min_j, int max_i, int max_j) override {
    switch (policy_) {
      case NAVO_TRUE_OVERWRITE: updateWithTrueOverwrite(master, min_i, min_j, max_i, max_j); break;
      case NAVO_OVERWRITE: updateWithOverwrite(master, min_i, min_j, max_i, max_j); break;
      case NAVO_MAX: updateWithMax(master, min_i, min_j, max_i, max_j); break;
      case NAVO_ADDITION: updateWithAddition(master, min_i, min_j, max_i, max_j); break;
      default: break;
    }
  }
  int policy_;
  unsigned x_, y_, width_, height_;
  bool has_updated_data_;
};

struct OwnedObservation {
  double ox, oy, oz, obstacle_range, raytrace_range;
  std::vector<float> xyz;
  bool marking, clearing;
};

// ObstacleLayer's algorithmic part on top of the reference's CostmapLayer primitives.
class RefObstacleLayer : public CostmapLayer {
 public:
  RefObstacleLayer(int combination_method, bool footprint_clearing, double max_obstacle_height)
      : combination_method_(combination_method),
        footprint_clearing_enabled_(footprint_clearing),
        max_obstacle_height_(max_obstacle_height),
        rolling_window_(false) {}
  void onInitialize() override {  // obstacle_layer.cpp:54-66
    rolling_window_ = layered_costmap_->isRolling();
    default_value_ = layered_costmap_->isTrackingUnknown() ? costmap_2d::NO_INFORMATION : costmap_2d::FREE_SPACE;
    matchSize();
    current_ = true;
    enabled_ = true;
  }
  void setEnabled(bool e) { enabled_ = e; }
  std::vector<OwnedObservation> observations_;

  void updateBounds(double robot_x, double robot_y, double robot_yaw, double* min_x, double* min_y, double* max_x,
                    double* max_y) override {  // obstacle_layer.cpp:340-413
    if (rolling_window_) updateOrigin(robot_x - getSizeInMetersX() / 2, robot_y - getSizeInMetersY() / 2);
    if (!enabled_) return;
    useExtraBounds(min_x, min_y, max_x, max_y);
    for (size_t i = 0; i < observations_.size(); ++i)
      if (observations_[i].clearing) raytraceFreespace(observations_[i], min_x, min_y, max_x, max_y);
    for (size_t k = 0; k < observations_.size(); ++k) {
      const OwnedObservation& obs = observations_[k];
      if (!obs.marking) continue;
      double sq_obstacle_range = obs.obstacle_range * obs.obstacle_range;
      for (size_t i = 0; i < obs.xyz.size() / 3; ++i) {
        double px = obs.xyz[3 * i], py = obs.xyz[3 * i + 1], pz = obs.xyz[3 * i + 2];
        if (pz > max_obstacle_height_) continue;
        double sq_dist = (px - obs.ox) * (px - obs.ox) + (py - obs.oy) * (py - obs.oy) + (pz - obs.oz) * (pz - obs.oz);
        if (sq_dist >= sq_obstacle_range) continue;
        unsigned int mx, my;
        if (!worldToMap(px, py, mx, my)) continue;
        costmap_[getIndex(mx, my)] = costmap_2d::LETHAL_OBSTACLE;
        touch(px, py, min_x, min_y, max_x, max_y);
      }
    }
    // updateFootprint, obstacle_layer.cpp:415-425
    if (!footprint_clearing_enabled_) return;
    costmap_2d::transformFootprint(robot_x, robot_y, robot_yaw, getFootprint(), transformed_footprint_);
    for (unsigned int i = 0; i < transformed_footprint_.size(); i++)
      touch(transformed_footprint_[i].x, transformed_footprint_[i].y, min_x, min_y, max_x, max_y);
  }

  void updateCosts(Costmap2D& master_grid, int min_i, int min_j, int max_i, int max_j) override {  // :427-448
    if (!enabled_) return;
    if (footprint_clearing_enabled_) setConvexPolygonCost(transformed_footprint_, costmap_2d::FREE_SPACE);
    switch (combination_method_) {
      case 0: updateWithOverwrite(master_grid, min_i, min_j, max_i, max_j); break;
      case 1: updateWithMax(master_grid, min_i, min_j, max_i, max_j); break;
      default: break;
    }
  }

 protected:
  void raytraceFreespace(const OwnedObservation& obs, double* min_x, double* min_y, double* max_x,
                         double* max_y) {  // obstacle_layer.cpp:498-576
    double ox = obs.ox, oy = obs.oy;
    unsigned int x0, y0;
    if (!worldToMap(ox, oy, x0, y0)) return;
    double origin_x = origin_x_, origin_y = origin_y_;
    double map_end_x = origin_x + size_x_ * resolution_;
    double map_end_y = origin_y + size_y_ * resolution_;
    touch(ox, oy, min_x, min_y, max_x, max_y);
    for (size_t i = 0; i < obs.xyz.size() / 3; ++i) {
      double wx = obs.xyz[3 * i];
      double wy = obs.xyz[3 * i + 1];
      double a = wx - ox;
      double b = wy - oy;
      if (wx < origin_x) {
        double t = (origin_x - ox) / a;
        wx = origin_x;
        wy = oy + b * t;
      }
      if (wy < origin_y) {
        double t = (origin_y - oy) / b;
        wx = ox + a * t;
        wy = origin_y;
      }
      if (wx > map_end_x) {
        double t = (map_end_x - ox) / a;
        wx = map_end_x - .001;
        wy = oy + b * t;
      }
      if (wy > map_end_y) {
        double t = (map_end_y - oy) / b;
        wx = ox + a * t;
        wy = map_end_y - .001;
      }
      unsigned int x1, y1;
      if (!worldToMap(wx, wy, x1, y1)) continue;
      unsigned int cell_raytrace_range = cellDistance(obs.raytrace_range);
      MarkCell marker(costmap_, costmap_2d::FREE_SPACE);
      raytraceLine(marker, x0, y0, x1, y1, cell_raytrace_range);
      // updateRaytraceBounds, obstacle_layer.cpp:602-610
      double dx = wx - ox, dy = wy - oy;
      double full_distance = hypot(dx, dy);
      double scale = std::min(1.0, obs.raytrace_range / full_distance);
      double ex = ox + dx * scale, ey = oy + dy * scale;
      touch(ex, ey, min_x, min_y, max_x, max_y);
    }
  }
  int combination_method_;
  bool footprint_clearing_enabled_;
  double max_obstacle_height_;
  bool rolling_window_;
  std::vector<geometry_msgs::Point> transformed_footprint_;
};


// VoxelLayer's algorithmic part (costmap_2d/plugins/voxel_layer.cpp) on top of the reference's own VoxelGrid and the
// ObstacleLayer restatement above (VoxelLayer derives from ObstacleLayer and inherits updateCosts).
class RefVoxelLayer : public RefObstacleLayer {
 public:
  RefVoxelLayer(int combination_method, bool footprint_clearing, double max_obstacle_height, double origin_z,
                double z_resolution, int z_voxels, int unknown_threshold, int mark_threshold)
      : RefObstacleLayer(combination_method, footprint_clearing, max_obstacle_height),
        voxel_grid_(0, 0, 0),
        z_resolution_(z_resolution),
        origin_z_(origin_z),
        unknown_threshold_(unknown_threshold + (VOXEL_BITS - z_voxels)),  // voxel_layer.cpp:92
        mark_threshold_(mark_threshold),
        size_z_(z_voxels) {}
  void matchSize() override {  // voxel_layer.cpp:97-102
    RefObstacleLayer::matchSize();
    voxel_grid_.resize(size_x_, size_y_, size_z_);
  }
  void resetMaps() override {  // :112-116
    Costmap2D::resetMaps();
    voxel_grid_.reset();
  }
  const uint32_t* voxels() { return voxel_grid_.getData(); }

  void updateBounds(double robot_x, double robot_y, double robot_yaw, double* min_x, double* min_y, double* max_x,
                    double* max_y) override {  // voxel_layer.cpp:116-177 (+ ObstacleLayer::updateFootprint :201)
    if (rolling_window_) updateOriginVoxel(robot_x - getSizeInMetersX() / 2, robot_y - getSizeInMetersY() / 2);
    if (!enabled_) return;
    useExtraBounds(min_x, min_y, max_x, max_y);
    for (size_t i = 0; i < observations_.size(); ++i)
      if (observations_[i].clearing) raytraceFreespaceVoxel(observations_[i], min_x, min_y, max_x, max_y);
    for (size_t k = 0; k < observations_.size(); ++k) {
      const OwnedObservation& obs = observations_[k];
      if (!obs.marking) continue;
      double sq_obstacle_range = obs.obstacle_range * obs.obstacle_range;
      for (size_t i = 0; i < obs.xyz.size() / 3; ++i) {
        const float fx = obs.xyz[3 * i], fy = obs.xyz[3 * i + 1], fz = obs.xyz[3 * i + 2];
        if (fz > max_obstacle_height_) continue;
        double sq_dist = (fx - obs.ox) * (fx - obs.ox) + (fy - obs.oy) * (fy - obs.oy) + (fz - obs.oz) * (fz - obs.oz);
        if (sq_dist >= sq_obstacle_range) continue;
        unsigned int mx, my, mz;
        if (fz < origin_z_) {
          if (!worldToMap3D(fx, fy, origin_z_, mx, my, mz)) continue;
        } else if (!worldToMap3D(fx, fy, fz, mx, my, mz)) {
          continue;
        }
        if (voxel_grid_.markVoxelInMap(mx, my, mz, mark_threshold_)) {
          costmap_[getIndex(mx, my)] = costmap_2d::LETHAL_OBSTACLE;
          touch((double)fx, (double)fy, min_x, min_y, max_x, max_y);
        }
      }
    }
    if (!footprint_clearing_enabled_) return;
    costmap_2d::transformFootprint(robot_x, robot_y, robot_yaw, getFootprint(), transformed_footprint_);
    for (unsigned int i = 0; i < transformed_footprint_.size(); i++)
      touch(transformed_footprint_[i].x, transformed_footprint_[i].y, min_x, min_y, max_x, max_y);
  }

 private:
  static const unsigned int VOXEL_BITS = 16;  // voxel_layer.cpp:44
  bool worldToMap3DFloat(double wx, double wy, double wz, double& mx, double& my, double& mz) {  // voxel_layer.h:103-115
    if (wx < origin_x_ || wy < origin_y_ || wz < origin_z_) return false;
    mx = ((wx - origin_x_) / resolution_);
    my = ((wy - origin_y_) / resolution_);
    mz = ((wz - origin_z_) / z_resolution_);
    return mx < size_x_ && my < size_y_ && mz < size_z_;
  }
  bool worldToMap3D(double wx, double wy, double wz, unsigned int& mx, unsigned int& my, unsigned int& mz) {  // :117-130
    if (wx < origin_x_ || wy < origin_y_ || wz < origin_z_) return false;
    mx = (int)((wx - origin_x_) / resolution_);
    my = (int)((wy - origin_y_) / resolution_);
    mz = (int)((wz - origin_z_) / z_resolution_);
    return mx < size_x_ && my < size_y_ && mz < size_z_;
  }
  static double dist3(double x0, double y0, double z0, double x1, double y1, double z1) {  // :140-143
    return sqrt((x1 - x0) * (x1 - x0) + (y1 - y0) * (y1 - y0) + (z1 - z0) * (z1 - z0));
  }
  void raytraceFreespaceVoxel(const OwnedObservation& obs, double* min_x, double* min_y, double* max_x,
                              double* max_y) {  // voxel_layer.cpp:262-350
    if (obs.xyz.empty()) return;
    double sensor_x, sensor_y, sensor_z;
    double ox = obs.ox, oy = obs.oy, oz = obs.oz;
    if (!worldToMap3DFloat(ox, oy, oz, sensor_x, sensor_y, sensor_z)) return;
    double map_end_x = origin_x_ + getSizeInMetersX();
    double map_end_y = origin_y_ + getSizeInMetersY();
    for (size_t i = 0; i < obs.xyz.size() / 3; ++i) {
      double wpx = obs.xyz[3 * i], wpy = obs.xyz[3 * i + 1], wpz = obs.xyz[3 * i + 2];
      double distance = dist3(ox, oy, oz, wpx, wpy, wpz);
      double scaling_fact = 1.0;
      scaling_fact = std::max(std::min(scaling_fact, (distance - 2 * resolution_) / distance), 0.0);
      wpx = scaling_fact * (wpx - ox) + ox;
      wpy = scaling_fact * (wpy - oy) + oy;
      wpz = scaling_fact * (wpz - oz) + oz;
      double a = wpx - ox, b = wpy - oy, c = wpz - oz, t = 1.0;
      if (wpz > max_obstacle_height_) {
        t = std::max(0.0, std::min(t, (max_obstacle_height_ - 0.01 - oz) / c));
      } else if (wpz < origin_z_) {
        t = std::min(t, (origin_z_ - oz) / c);
      }
      if (wpx < origin_x_) t = std::min(t, (origin_x_ - ox) / a);
      if (wpy < origin_y_) t = std::min(t, (origin_y_ - oy) / b);
      if (wpx > map_end_x) t = std::min(t, (map_end_x - ox) / a);
      if (wpy > map_end_y) t = std::min(t, (map_end_y - oy) / b);
      wpx = ox + a * t;
      wpy = oy + b * t;
      wpz = oz + c * t;
      double point_x, point_y, point_z;
      if (worldToMap3DFloat(wpx, wpy, wpz, point_x, point_y, point_z)) {
        unsigned int cell_raytrace_range = cellDistance(obs.raytrace_range);
        voxel_grid_.clearVoxelLineInMap(sensor_x, sensor_y, sensor_z, point_x, point_y, point_z, costmap_,
                                        unknown_threshold_, mark_threshold_, costmap_2d::FREE_SPACE,
                                        costmap_2d::NO_INFORMATION, cell_raytrace_range);
        // updateRaytraceBounds, obstacle_layer.cpp:602-610
        double dx = wpx - ox, dy = wpy - oy;
        double full_distance = hypot(dx, dy);
        double scale = std::min(1.0, obs.raytrace_range / full_distance);
        touch(ox + dx * scale, oy + dy * scale, min_x, min_y, max_x, max_y);
      }
    }
  }
  void updateOriginVoxel(double new_origin_x, double new_origin_y) {  // voxel_layer.cpp:371-438
    int cell_ox = int((new_origin_x - origin_x_) / resolution_), cell_oy = int((new_origin_y - origin_y_) / resolution_);
    double new_grid_ox = origin_x_ + cell_ox * resolution_, new_grid_oy = origin_y_ + cell_oy * resolution_;
    int size_x = size_x_, size_y = size_y_;
    int lower_left_x = std::min(std::max(cell_ox, 0), size_x), lower_left_y = std::min(std::max(cell_oy, 0), size_y);
    int upper_right_x = std::min(std::max(cell_ox + size_x, 0), size_x);
    int upper_right_y = std::min(std::max(cell_oy + size_y, 0), size_y);
    unsigned int cell_size_x = upper_right_x - lower_left_x, cell_size_y = upper_right_y - lower_left_y;
    unsigned char* local_map = new unsigned char[cell_size_x * cell_size_y];
    unsigned int* local_voxel_map = new unsigned int[cell_size_x * cell_size_y];
    unsigned int* voxel_map = voxel_grid_.getData();
    copyMapRegion(costmap_, lower_left_x, lower_left_y, size_x_, local_map, 0, 0, cell_size_x, cell_size_x, cell_size_y);
    copyMapRegion(voxel_map, lower_left_x, lower_left_y, size_x_, local_voxel_map, 0, 0, cell_size_x, cell_size_x, cell_size_y);
    resetMaps();
    origin_x_ = new_grid_ox;
    origin_y_ = new_grid_oy;
    int start_x = lower_left_x - cell_ox, start_y = lower_left_y - cell_oy;
    copyMapRegion(local_map, 0, 0, cell_size_x, costmap_, start_x, start_y, size_x_, cell_size_x, cell_size_y);
    copyMapRegion(local_voxel_map, 0, 0, cell_size_x, voxel_map, start_x, start_y, size_x_, cell_size_x, cell_size_y);
    delete[] local_map;
    delete[] local_voxel_map;
  }
  voxel_grid::VoxelGrid voxel_grid_;
  double z_resolution_, origin_z_;
  unsigned int unknown_threshold_, mark_threshold_, size_z_;
};

// exposes Costmap2D's protected raytraceLine
class RayProbe : public Costmap2D {
 public:
  RayProbe(unsigned sx) : Costmap2D(sx, 1, 1.0, 0, 0) {}
  struct Collect {
    std::vector<unsigned>* v;
    void operator()(unsigned off) { v->push_back(off); }
  };
  void trace(unsigned x0, unsigned y0, unsigned x1, unsigned y1, unsigned maxlen, std::vector<unsigned>& out) {
    Collect c{&out};
    raytraceLine(c, x0, y0, x1, y1, maxlen);
  }
};

struct CostmapHandle {
  std::unique_ptr<LayeredCostmap> lc;
  std::vector<costmap_2d::Layer*> layers;  // owned by lc's shared_ptrs
  std::vector<int> kinds;                  // 0 grid, 1 obstacle, 2 inflation
  std::vector<double> infl_radius;         // per layer (only meaningful for kind 2)
  tf::TransformListener tf;
};

std::vector<geometry_msgs::Point> toPoints(const double* xy, int n) {
  std::vector<geometry_msgs::Point> v(n);
  for (int i = 0; i < n; ++i) {
    v[i].x = xy[2 * i];
    v[i].y = xy[2 * i + 1];
  }
  return v;
}

}  // namespace

extern "C" {

const char* navo_impl_name(void) { return "reference"; }

void* navo_costmap_create(uint32_t size_x, uint32_t size_y, double resolution, double origin_x, double origin_y,
                          int rolling_window, int track_unknown) {
  CostmapHandle* h = new CostmapHandle;
  h->lc.reset(new LayeredCostmap("map", rolling_window != 0, track_unknown != 0));
  h->lc->resizeMap(size_x, size_y, resolution, origin_x, origin_y);
  return h;
}
void navo_costmap_destroy(void* hv) { delete static_cast<CostmapHandle*>(hv); }

static int addLayer(CostmapHandle* h, costmap_2d::Layer* l, int kind, const char* name) {
  h->lc->addPlugin(boost::shared_ptr<costmap_2d::Layer>(l));
  l->initialize(h->lc.get(), name, &h->tf);
  h->layers.push_back(l);
  h->kinds.push_back(kind);
  h->infl_radius.push_back(0.0);
  return int(h->layers.size()) - 1;
}
int navo_costmap_add_grid_layer(void* hv, int policy) {
  return addLayer(static_cast<CostmapHandle*>(hv), new GridLayer(policy), 0, "grid");
}
int navo_costmap_add_obstacle_layer(void* hv, int combination_method, int footprint_clearing,
                                    double max_obstacle_height) {
  return addLayer(static_cast<CostmapHandle*>(hv),
                  new RefObstacleLayer(combination_method, footprint_clearing != 0, max_obstacle_height), 1,
                  "obstacles");
}
int navo_costmap_add_voxel_layer(void* hv, int combination_method, int footprint_clearing, double max_obstacle_height,
                                 double origin_z, double z_resolution, int z_voxels, int unknown_threshold,
                                 int mark_threshold) {
  // kind 1: everything the C API does with an obstacle layer applies (observations, enable, grid read-back)
  return addLayer(static_cast<CostmapHandle*>(hv),
                  new RefVoxelLayer(combination_method, footprint_clearing != 0, max_obstacle_height, origin_z,
                                    z_resolution, z_voxels, unknown_threshold, mark_threshold), 1, "voxels");
}
void navo_layer_get_voxels(void* hv, int layer, uint32_t* out) {
  CostmapHandle* h = static_cast<CostmapHandle*>(hv);
  RefVoxelLayer* v = dynamic_cast<RefVoxelLayer*>(h->layers[layer]);
  if (!v) return;
  Costmap2D* c = h->lc->getCostmap();
  memcpy(out, v->voxels(), size_t(c->getSizeInCellsX()) * c->getSizeInCellsY() * sizeof(uint32_t));
}
namespace {
struct VoxelCollect {  // an ActionType for the reference's VoxelGrid::raytraceLine template
  std::vector<std::pair<unsigned, unsigned> >* v;
  void operator()(unsigned int offset, unsigned int z_mask) { v->push_back(std::make_pair(offset, z_mask)); }
};
}  // namespace
int navo_voxel_line_cells(uint32_t size_x, double x0, double y0, double z0, double x1, double y1, double z1,
                          uint32_t max_length, uint32_t* offsets_out, int32_t* z_out, int capacity) {
  unsigned size_y = unsigned(std::max(y0, y1)) + 2;
  voxel_grid::VoxelGrid vg(size_x, size_y, 16);
  std::vector<std::pair<unsigned, unsigned> > cells;
  VoxelCollect c{&cells};
  vg.raytraceLine(c, x0, y0, z0, x1, y1, z1, max_length);
  int n = 0;
  for (size_t i = 0; i < cells.size() && n < capacity; ++i, ++n) {
    offsets_out[n] = cells[i].first;
    z_out[n] = __builtin_ctz(cells[i].second & 0xffffu ? cells[i].second & 0xffffu : 0x10000u);
  }
  return int(cells.size());
}
int navo_costmap_add_inflation_layer(void* hv, double inflation_radius, double cost_scaling_factor) {
  CostmapHandle* h = static_cast<CostmapHandle*>(hv);
  costmap_2d::InflationLayer* il = new costmap_2d::InflationLayer();
  int id = addLayer(h, il, 2, "inflation");
  il->setInflationParameters(inflation_radius, cost_scaling_factor);
  h->infl_radius[id] = inflation_radius;
  return id;
}
void navo_costmap_set_footprint(void* hv, const double* xy, int n) {
  static_cast<CostmapHandle*>(hv)->lc->setFootprint(toPoints(xy, n));
}
void navo_grid_layer_set(void* hv, int layer, const uint8_t* data) {
  static_cast<GridLayer*>(static_cast<CostmapHandle*>(hv)->layers[layer])->setData(data);
}
void navo_grid_layer_touch(void* hv, int layer, uint32_t x, uint32_t y, uint32_t w, uint32_t hgt) {
  static_cast<GridLayer*>(static_cast<CostmapHandle*>(hv)->layers[layer])->touchRegion(x, y, w, hgt);
}
void navo_layer_set_enabled(void* hv, int layer, int enabled) {
  CostmapHandle* h = static_cast<CostmapHandle*>(hv);
  if (h->kinds[layer] == 0) static_cast<GridLayer*>(h->layers[layer])->setEnabled(enabled != 0);
  if (h->kinds[layer] == 1) static_cast<RefObstacleLayer*>(h->layers[layer])->setEnabled(enabled != 0);
}
void navo_obstacle_set_observations(void* hv, int layer, const navo_observation* obs, int n_obs) {
  RefObstacleLayer* ol = static_cast<RefObstacleLayer*>(static_cast<CostmapHandle*>(hv)->layers[layer]);
  ol->observations_.clear();
  for (int i = 0; i < n_obs; ++i) {
    OwnedObservation o;
    o.ox = obs[i].origin_x; o.oy = obs[i].origin_y; o.oz = obs[i].origin_z;
    o.obstacle_range = obs[i].obstacle_range;
    o.raytrace_range = obs[i].raytrace_range;
    o.xyz.assign(obs[i].xyz, obs[i].xyz + 3 * size_t(obs[i].n_points));
    o.marking = obs[i].marking != 0;
    o.clearing = obs[i].clearing != 0;
    ol->observations_.push_back(o);
  }
}
void navo_inflation_set_params(void* hv, int layer, double inflation_radius, double cost_scaling_factor) {
  static_cast<CostmapHandle*>(hv)->infl_radius[layer] = inflation_radius;
  static_cast<costmap_2d::InflationLayer*>(static_cast<CostmapHandle*>(hv)->layers[layer])
      ->setInflationParameters(inflation_radius, cost_scaling_factor);
}
// the compiled reference has exactly one behaviour: libstdc++'s heap order (variant 0)
int navo_inflation_set_variant(void*, int, int variant, uint64_t) { return variant == 0 ? 0 : -1; }
int navo_inflation_last_rounds(void*, int) { return 0; }
void navo_costmap_update_map(void* hv, double rx, double ry, double ryaw, int32_t w[4]) {
  CostmapHandle* h = static_cast<CostmapHandle*>(hv);
  h->lc->updateMap(rx, ry, ryaw);
  unsigned int x0, xn, y0, yn;
  h->lc->getBounds(&x0, &xn, &y0, &yn);
  w[0] = x0; w[1] = xn; w[2] = y0; w[3] = yn;
}
void navo_costmap_get(void* hv, uint8_t* out) {
  Costmap2D* c = static_cast<CostmapHandle*>(hv)->lc->getCostmap();
  memcpy(out, c->getCharMap(), size_t(c->getSizeInCellsX()) * c->getSizeInCellsY());
}
void navo_costmap_set(void* hv, const uint8_t* in) {
  Costmap2D* c = static_cast<CostmapHandle*>(hv)->lc->getCostmap();
  memcpy(c->getCharMap(), in, size_t(c->getSizeInCellsX()) * c->getSizeInCellsY());
}
void navo_layer_get(void* hv, int layer, uint8_t* out) {
  CostmapHandle* h = static_cast<CostmapHandle*>(hv);
  if (h->kinds[layer] == 2) return;
  Costmap2D* c = (h->kinds[layer] == 0) ? static_cast<Costmap2D*>(static_cast<GridLayer*>(h->layers[layer]))
                                        : static_cast<Costmap2D*>(static_cast<RefObstacleLayer*>(h->layers[layer]));
  memcpy(out, c->getCharMap(), size_t(c->getSizeInCellsX()) * c->getSizeInCellsY());
}
void navo_costmap_get_origin(void* hv, double out[2]) {
  Costmap2D* c = static_cast<CostmapHandle*>(hv)->lc->getCostmap();
  out[0] = c->getOriginX();
  out[1] = c->getOriginY();
}
int navo_inflation_tables(void* hv, int layer, uint8_t* costs_out, double* dists_out, int capacity) {
  // The cached tables are private; they are fully determined by the public computeCost and hypot, exactly as
  // computeCaches builds them (inflation_layer.cpp:295-328); R as matchSize computes it (:110-123).
  CostmapHandle* h = static_cast<CostmapHandle*>(hv);
  costmap_2d::InflationLayer* il = static_cast<costmap_2d::InflationLayer*>(h->layers[layer]);
  int R = int(h->lc->getCostmap()->cellDistance(h->infl_radius[layer]));
  int n = R + 2;
  if (n * n > capacity) return R;
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      double d = hypot(i, j);
      dists_out[i * n + j] = d;
      costs_out[i * n + j] = il->computeCost(d);
    }
  return R;
}

void navo_interpret_values(const uint8_t* in, uint8_t* out, int64_t n, int track_unknown, uint8_t unknown_cost_value,
                           uint8_t lethal_threshold, int trinary) {  // static_layer.cpp:149-163
  for (int64_t i = 0; i < n; ++i) {
    unsigned char value = in[i];
    unsigned char r;
    if (track_unknown && value == unknown_cost_value) r = costmap_2d::NO_INFORMATION;
    else if (!track_unknown && value == unknown_cost_value) r = costmap_2d::FREE_SPACE;
    else if (value >= lethal_threshold) r = costmap_2d::LETHAL_OBSTACLE;
    else if (trinary) r = costmap_2d::FREE_SPACE;
    else {
      double scale = (double)value / lethal_threshold;
      r = scale * costmap_2d::LETHAL_OBSTACLE;
    }
    out[i] = r;
  }
}

int navo_raytrace_cells(uint32_t size_x, uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1, uint32_t max_length,
                        uint32_t* offsets_out, int capacity) {
  RayProbe p(size_x);
  std::vector<unsigned> v;
  p.trace(x0, y0, x1, y1, max_length, v);
  for (size_t i = 0; i < v.size() && int(i) < capacity; ++i) offsets_out[i] = v[i];
  return int(v.size());
}

void navo_footprint_radii(const double* xy, int n, double* inscribed, double* circumscribed) {
  costmap_2d::calculateMinAndMaxDistances(toPoints(xy, n), *inscribed, *circumscribed);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ Path B
namespace {

using namespace base_local_planner;

std::vector<geometry_msgs::PoseStamped> toPoses(const double* xy, int n) {
  std::vector<geometry_msgs::PoseStamped> v(n);
  for (int i = 0; i < n; ++i) {
    v[i].pose.position.x = xy[2 * i];
    v[i].pose.position.y = xy[2 * i + 1];
  }
  return v;
}

// DWAPlanner's wiring (dwa_planner.cpp:116-182) around the reference's critics / generator / search.
struct DwaHandle {
  navo_dwa_config cfg;
  Costmap2D costmap;
  LocalPlannerLimits limits;
  ObstacleCostFunction obstacle_costs_;
  MapGridCostFunction path_costs_, goal_costs_, goal_front_costs_, alignment_costs_;
  OscillationCostFunction oscillation_costs_;
  SimpleTrajectoryGenerator generator_;
  SimpleScoredSamplingPlanner scored_sampling_planner_;
  std::vector<geometry_msgs::PoseStamped> global_plan_;
  Eigen::Vector3f vsamples_;
  double pdist_scale_, gdist_scale_, occdist_scale_, forward_point_distance_, cheat_factor_;
  Trajectory result_traj_;

  DwaHandle(const navo_dwa_config& c, unsigned sx, unsigned sy, double res)
      : cfg(c),
        costmap(sx, sy, res, 0.0, 0.0, 0),
        obstacle_costs_(&costmap),
        path_costs_(&costmap),
        goal_costs_(&costmap, 0.0, 0.0, true),
        goal_front_costs_(&costmap, 0.0, 0.0, true),
        alignment_costs_(&costmap) {
    goal_front_costs_.setStopOnFailure(false);
    alignment_costs_.setStopOnFailure(false);
    oscillation_costs_.resetOscillationFlags();
    obstacle_costs_.setSumScores(c.sum_scores != 0);
    std::vector<TrajectoryCostFunction*> critics;
    critics.push_back(&oscillation_costs_);
    critics.push_back(&obstacle_costs_);
    critics.push_back(&goal_front_costs_);
    critics.push_back(&alignment_costs_);
    critics.push_back(&path_costs_);
    critics.push_back(&goal_costs_);
    std::vector<TrajectorySampleGenerator*> generator_list;
    generator_list.push_back(&generator_);
    scored_sampling_planner_ = SimpleScoredSamplingPlanner(generator_list, critics);
    cheat_factor_ = c.cheat_factor;
    reconfigure();
  }
  void reconfigure() {  // dwa_planner.cpp:52-112
    const navo_dwa_config& c = cfg;
    limits.max_trans_vel = c.max_trans_vel; limits.min_trans_vel = c.min_trans_vel;
    limits.max_vel_x = c.max_vel_x; limits.min_vel_x = c.min_vel_x;
    limits.max_vel_y = c.max_vel_y; limits.min_vel_y = c.min_vel_y;
    limits.max_rot_vel = c.max_rot_vel; limits.min_rot_vel = c.min_rot_vel;
    limits.acc_lim_x = c.acc_lim_x; limits.acc_lim_y = c.acc_lim_y; limits.acc_lim_theta = c.acc_lim_theta;
    generator_.setParameters(c.sim_time, c.sim_granularity, c.angular_sim_granularity, c.use_dwa != 0, c.sim_period);
    double resolution = costmap.getResolution();
    pdist_scale_ = c.path_distance_bias;
    path_costs_.setScale(resolution * pdist_scale_ * 0.5);
    alignment_costs_.setScale(resolution * pdist_scale_ * 0.5);
    gdist_scale_ = c.goal_distance_bias;
    goal_costs_.setScale(resolution * gdist_scale_ * 0.5);
    goal_front_costs_.setScale(resolution * gdist_scale_ * 0.5);
    occdist_scale_ = c.occdist_scale;
    obstacle_costs_.setScale(resolution * occdist_scale_);
    oscillation_costs_.setOscillationResetDist(c.oscillation_reset_dist, c.oscillation_reset_angle);
    forward_point_distance_ = c.forward_point_distance;
    goal_front_costs_.setXShift(forward_point_distance_);
    alignment_costs_.setXShift(forward_point_distance_);
    obstacle_costs_.setParams(c.max_trans_vel, c.max_scaling_factor, c.scaling_speed);
    int vx = c.vx_samples <= 0 ? 1 : c.vx_samples;
    int vy = c.vy_samples <= 0 ? 1 : c.vy_samples;
    int vth = c.vth_samples <= 0 ? 1 : c.vth_samples;
    vsamples_[0] = vx; vsamples_[1] = vy; vsamples_[2] = vth;
  }
};

// Costmap2D keeps its origin protected; this subclass-free trick re-creates geometry through resizeMap.
void setCostmap(Costmap2D& cm, const uint8_t* grid, double ox, double oy) {
  unsigned sx = cm.getSizeInCellsX(), sy = cm.getSizeInCellsY();
  if (cm.getOriginX() != ox || cm.getOriginY() != oy) {
    // updateOrigin snaps to the grid; resizeMap sets the origin verbatim and keeps the same buffer size
    cm.resizeMap(sx, sy, cm.getResolution(), ox, oy);
  }
  memcpy(cm.getCharMap(), grid, size_t(sx) * sy);
}

}  // namespace

extern "C" {

void navo_dwa_default_config(navo_dwa_config* c) {
  // base_local_planner/src/local_planner_limits/__init__.py:15-45, dwa_local_planner/cfg/DWAPlanner.cfg:15-43
  c->max_trans_vel = 0.55; c->min_trans_vel = 0.1; c->max_vel_x = 0.55; c->min_vel_x = 0.0;
  c->max_vel_y = 0.1; c->min_vel_y = -0.1; c->max_rot_vel = 1.0; c->min_rot_vel = 0.4;
  c->acc_lim_x = 2.5; c->acc_lim_y = 2.5; c->acc_lim_theta = 3.2;
  c->sim_time = 1.7; c->sim_granularity = 0.025; c->angular_sim_granularity = 0.1; c->sim_period = 0.05;
  c->path_distance_bias = 32.0; c->goal_distance_bias = 24.0; c->occdist_scale = 0.01;
  c->forward_point_distance = 0.325; c->cheat_factor = 1.0;
  c->oscillation_reset_dist = 0.05; c->oscillation_reset_angle = 0.2;
  c->scaling_speed = 0.25; c->max_scaling_factor = 0.2;
  c->vx_samples = 3; c->vy_samples = 10; c->vth_samples = 20;
  c->use_dwa = 1; c->sum_scores = 0; c->allow_unknown = 0;
}

void* navo_dwa_create(const navo_dwa_config* cfg, uint32_t size_x, uint32_t size_y, double resolution) {
  return new DwaHandle(*cfg, size_x, size_y, resolution);
}
void navo_dwa_destroy(void* hv) { delete static_cast<DwaHandle*>(hv); }
void navo_dwa_reconfigure(void* hv, const navo_dwa_config* cfg) {
  DwaHandle* h = static_cast<DwaHandle*>(hv);
  h->cfg = *cfg;
  // the two construction parameters that navo_dwa_config carries (dwa_planner.cpp:116-182) follow cfg too
  h->cheat_factor_ = cfg->cheat_factor;
  h->obstacle_costs_.setSumScores(cfg->sum_scores != 0);
  h->reconfigure();
}
void navo_dwa_set_costmap(void* hv, const uint8_t* grid, double ox, double oy) {
  setCostmap(static_cast<DwaHandle*>(hv)->costmap, grid, ox, oy);
}

void navo_dwa_set_plan(void* hv, const double pose[3], const double* plan_xy, int n) {  // dwa_planner.cpp:240-286
  DwaHandle* h = static_cast<DwaHandle*>(hv);
  h->global_plan_ = toPoses(plan_xy, n);
  h->path_costs_.setTargetPoses(h->global_plan_);
  h->goal_costs_.setTargetPoses(h->global_plan_);
  geometry_msgs::PoseStamped goal_pose = h->global_plan_.back();
  Eigen::Vector3f pos(pose[0], pose[1], pose[2]);
  double sq_dist = (pos[0] - goal_pose.pose.position.x) * (pos[0] - goal_pose.pose.position.x) +
                   (pos[1] - goal_pose.pose.position.y) * (pos[1] - goal_pose.pose.position.y);
  std::vector<geometry_msgs::PoseStamped> front_global_plan = h->global_plan_;
  double angle_to_goal = atan2(goal_pose.pose.position.y - pos[1], goal_pose.pose.position.x - pos[0]);
  front_global_plan.back().pose.position.x =
      front_global_plan.back().pose.position.x + h->forward_point_distance_ * cos(angle_to_goal);
  front_global_plan.back().pose.position.y =
      front_global_plan.back().pose.position.y + h->forward_point_distance_ * sin(angle_to_goal);
  h->goal_front_costs_.setTargetPoses(front_global_plan);
  if (sq_dist > h->forward_point_distance_ * h->forward_point_distance_ * h->cheat_factor_) {
    double resolution = h->costmap.getResolution();
    h->alignment_costs_.setScale(resolution * h->pdist_scale_ * 0.5);
    h->alignment_costs_.setTargetPoses(h->global_plan_);
  } else {
    h->alignment_costs_.setScale(0.0);
  }
}

void navo_dwa_reset_oscillation(void* hv) { static_cast<DwaHandle*>(hv)->oscillation_costs_.resetOscillationFlags(); }

int navo_dwa_get_oscillation_mask(void* hv) {
  // the *_only_ flags are private; probe them through the public scoreTrajectory (oscillation_cost_function.cpp:166-176)
  DwaHandle* h = static_cast<DwaHandle*>(hv);
  const double probes[6][3] = {{-1, 0, 0}, {1, 0, 0}, {0, -1, 0}, {0, 1, 0}, {0, 0, -1}, {0, 0, 1}};
  int mask = 0;
  for (int i = 0; i < 6; ++i) {
    Trajectory t;
    t.xv_ = probes[i][0]; t.yv_ = probes[i][1]; t.thetav_ = probes[i][2];
    if (h->oscillation_costs_.scoreTrajectory(t) < 0) mask |= 1 << i;
  }
  return mask;
}

int navo_dwa_find_best_path(void* hv, const double pose[3], const double velv[3], const double* footprint_xy,
                            int n_footprint, navo_dwa_result* result, double* all_costs, int all_capacity,
                            double* best_points, int points_capacity) {  // dwa_planner.cpp:292-371
  DwaHandle* h = static_cast<DwaHandle*>(hv);
  h->obstacle_costs_.setFootprint(toPoints(footprint_xy, n_footprint));
  Eigen::Vector3f pos(pose[0], pose[1], pose[2]);
  Eigen::Vector3f vel(velv[0], velv[1], velv[2]);
  geometry_msgs::PoseStamped goal_pose = h->global_plan_.back();
  Eigen::Vector3f goal(goal_pose.pose.position.x, goal_pose.pose.position.y, 0.0f);
  LocalPlannerLimits limits = h->limits;
  h->generator_.initialise(pos, vel, goal, &limits, h->vsamples_);
  h->result_traj_.cost_ = -7;
  std::vector<Trajectory> all_explored;
  h->scored_sampling_planner_.findBestTrajectory(h->result_traj_, &all_explored);

  // Recover per-sample bookkeeping: re-enumerate the samples exactly as the generator did, and walk all_explored
  // (which holds only samples whose generateTrajectory succeeded, in order).
  h->generator_.initialise(pos, vel, goal, &limits, h->vsamples_);
  int n_samples = 0, k = 0, best_index = -1;
  bool best_found = false;
  while (h->generator_.hasMoreTrajectories()) {
    Trajectory t;
    bool ok = h->generator_.nextTrajectory(t);
    double c = std::numeric_limits<double>::quiet_NaN();
    if (ok) {
      c = all_explored[k].cost_;
      // the winner is the first sample whose reported cost equals the final best cost with identical velocities
      if (!best_found && h->result_traj_.cost_ >= 0 && c == h->result_traj_.cost_ &&
          all_explored[k].xv_ == h->result_traj_.xv_ && all_explored[k].yv_ == h->result_traj_.yv_ &&
          all_explored[k].thetav_ == h->result_traj_.thetav_) {
        best_index = n_samples;
        best_found = true;
      }
      ++k;
    }
    if (all_costs && n_samples < all_capacity) all_costs[n_samples] = c;
    ++n_samples;
  }
  h->oscillation_costs_.updateOscillationFlags(pos, &h->result_traj_, limits.min_trans_vel);

  result->cost = h->result_traj_.cost_;
  result->xv = h->result_traj_.xv_;
  result->yv = h->result_traj_.yv_;
  result->thetav = h->result_traj_.thetav_;
  result->best_index = best_index;
  result->n_samples = n_samples;
  result->n_scored = int(all_explored.size());
  result->n_points = int(h->result_traj_.getPointsSize());
  if (best_points) {
    for (unsigned i = 0; i < h->result_traj_.getPointsSize() && int(i) < points_capacity; ++i)
      h->result_traj_.getPoint(i, best_points[3 * i], best_points[3 * i + 1], best_points[3 * i + 2]);
  }
  return h->result_traj_.cost_ >= 0 ? 1 : 0;
}

double navo_dwa_check_trajectory(void* hv, const double pose[3], const double velv[3], const double vel_samples[3],
                                 const double* footprint_xy, int n_footprint) {  // dwa_planner.cpp:213-237
  DwaHandle* h = static_cast<DwaHandle*>(hv);
  h->obstacle_costs_.setFootprint(toPoints(footprint_xy, n_footprint));  // what the last findBestPath left behind
  Eigen::Vector3f pos(pose[0], pose[1], pose[2]);
  Eigen::Vector3f vel(velv[0], velv[1], velv[2]);
  Eigen::Vector3f samp(vel_samples[0], vel_samples[1], vel_samples[2]);
  h->oscillation_costs_.resetOscillationFlags();
  Trajectory traj;
  geometry_msgs::PoseStamped goal_pose = h->global_plan_.back();
  Eigen::Vector3f goal(goal_pose.pose.position.x, goal_pose.pose.position.y, 0.0f);
  LocalPlannerLimits limits = h->limits;
  h->generator_.initialise(pos, vel, goal, &limits, h->vsamples_);
  h->generator_.generateTrajectory(pos, vel, samp, traj);
  return h->scored_sampling_planner_.scoreTrajectory(traj, -1);
}

void navo_dwa_get_grid(void* hv, int which, double* out) {
  DwaHandle* h = static_cast<DwaHandle*>(hv);
  MapGridCostFunction* g[4] = {&h->path_costs_, &h->goal_costs_, &h->goal_front_costs_, &h->alignment_costs_};
  unsigned sx = h->costmap.getSizeInCellsX(), sy = h->costmap.getSizeInCellsY();
  for (unsigned y = 0; y < sy; ++y)
    for (unsigned x = 0; x < sx; ++x) out[size_t(y) * sx + x] = g[which]->getCellCosts(x, y);
}

void navo_dwa_prepare_only(void* hv) {
  DwaHandle* h = static_cast<DwaHandle*>(hv);
  h->goal_front_costs_.prepare();
  h->alignment_costs_.prepare();
  h->path_costs_.prepare();
  h->goal_costs_.prepare();
}

int navo_velocity_samples(double vmin, double vmax, int num_samples, double* out, int capacity) {
  VelocityIterator it(vmin, vmax, num_samples);
  int n = 0;
  for (; !it.isFinished(); it++) {
    if (n < capacity) out[n] = it.getVelocity();
    ++n;
  }
  return n;
}

int navo_line_cells(int x0, int y0, int x1, int y1, int32_t* xy_out, int capacity) {
  int n = 0;
  for (LineIterator line(x0, y0, x1, y1); line.isValid(); line.advance()) {
    if (n < capacity) {
      xy_out[2 * n] = line.getX();
      xy_out[2 * n + 1] = line.getY();
    }
    ++n;
  }
  return n;
}

void navo_mapgrid_bfs(const uint8_t* costs, uint32_t size_x, uint32_t size_y, const int32_t* seeds_xy, int n_seeds,
                      int /*allow_unknown*/, double* dist_out) {
  // as base_local_planner/test/utest.cpp:104-166 drives it
  Costmap2D cm(size_x, size_y, 1.0, 0.0, 0.0, 0);
  memcpy(cm.getCharMap(), costs, size_t(size_x) * size_y);
  MapGrid mg(size_x, size_y);
  mg.resetPathDist();
  std::queue<MapCell*> q;
  for (int i = 0; i < n_seeds; ++i) {
    MapCell& c = mg.getCell(seeds_xy[2 * i], seeds_xy[2 * i + 1]);
    c.target_dist = 0.0;
    c.target_mark = true;
    q.push(&c);
  }
  mg.computeTargetDistance(q, cm);
  for (uint32_t y = 0; y < size_y; ++y)
    for (uint32_t x = 0; x < size_x; ++x) dist_out[size_t(y) * size_x + x] = mg(x, y).target_dist;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// legacy TrajectoryPlanner: the reference's own class, constructed as TrajectoryPlannerROS::initialize does
// (trajectory_planner_ros.cpp:116-250) and driven through its public findBestPath / scoreTrajectory.
namespace {
struct TpHandle {
  Costmap2D costmap;
  CostmapModel world_model;
  std::unique_ptr<TrajectoryPlanner> tp;
  TpHandle(const navo_tp_config& c, unsigned sx, unsigned sy, double res, const double* fp, int nfp)
      : costmap(sx, sy, res, 0.0, 0.0, 0), world_model(costmap) {
    std::vector<double> yv(c.y_vels, c.y_vels + c.n_y_vels);
    tp.reset(new TrajectoryPlanner(world_model, costmap, toPoints(fp, nfp), c.acc_lim_x, c.acc_lim_y, c.acc_lim_theta,
                                   c.sim_time, c.sim_granularity, c.vx_samples, c.vtheta_samples, c.pdist_scale,
                                   c.gdist_scale, c.occdist_scale, c.heading_lookahead, c.oscillation_reset_dist,
                                   c.escape_reset_dist, c.escape_reset_theta, c.holonomic_robot != 0, c.max_vel_x,
                                   c.min_vel_x, c.max_vel_th, c.min_vel_th, c.min_in_place_vel_th, c.backup_vel,
                                   c.dwa != 0, c.heading_scoring != 0, c.heading_scoring_timestep, false,
                                   c.simple_attractor != 0, yv, c.stop_time_buffer, c.sim_period,
                                   c.angular_sim_granularity));
  }
};
}  // namespace

extern "C" {

void navo_tp_default_config(navo_tp_config* c) {
  memset(c, 0, sizeof(*c));
  c->acc_lim_x = 2.5; c->acc_lim_y = 2.5; c->acc_lim_theta = 3.2;
  c->sim_time = 1.0; c->sim_granularity = 0.025; c->angular_sim_granularity = 0.025; c->sim_period = 0.05;
  c->pdist_scale = 0.6; c->gdist_scale = 0.8; c->occdist_scale = 0.01;
  c->heading_lookahead = 0.325; c->oscillation_reset_dist = 0.05; c->escape_reset_dist = 0.10;
  c->escape_reset_theta = M_PI_4;
  c->max_vel_x = 0.5; c->min_vel_x = 0.1; c->max_vel_th = 1.0; c->min_vel_th = -1.0; c->min_in_place_vel_th = 0.4;
  c->backup_vel = -0.1; c->heading_scoring_timestep = 0.8; c->stop_time_buffer = 0.2;
  c->y_vels[0] = -0.3; c->y_vels[1] = -0.1; c->y_vels[2] = 0.1; c->y_vels[3] = 0.3; c->n_y_vels = 4;
  c->vx_samples = 3; c->vtheta_samples = 20;
  c->holonomic_robot = 1; c->dwa = 1; c->heading_scoring = 0; c->simple_attractor = 0; c->allow_unknown = 0;
}

void* navo_tp_create(const navo_tp_config* cfg, uint32_t size_x, uint32_t size_y, double resolution,
                     const double* footprint_xy, int n_footprint) {
  return new TpHandle(*cfg, size_x, size_y, resolution, footprint_xy, n_footprint);
}
void navo_tp_destroy(void* hv) { delete static_cast<TpHandle*>(hv); }
void navo_tp_reconfigure(void* hv, const navo_tp_config* c) {
  TpHandle* h = static_cast<TpHandle*>(hv);
  base_local_planner::BaseLocalPlannerConfig config;  // what TrajectoryPlannerROS::reconfigureCB hands over (trajectory_planner_ros.cpp)
  config.acc_lim_x = c->acc_lim_x; config.acc_lim_y = c->acc_lim_y; config.acc_lim_theta = c->acc_lim_theta;
  config.max_vel_x = c->max_vel_x; config.min_vel_x = c->min_vel_x;
  config.max_vel_theta = c->max_vel_th; config.min_vel_theta = c->min_vel_th;
  config.min_in_place_vel_theta = c->min_in_place_vel_th;
  config.sim_time = c->sim_time; config.sim_granularity = c->sim_granularity;
  config.angular_sim_granularity = c->angular_sim_granularity;
  config.pdist_scale = c->pdist_scale; config.gdist_scale = c->gdist_scale; config.occdist_scale = c->occdist_scale;
  config.oscillation_reset_dist = c->oscillation_reset_dist; config.escape_reset_dist = c->escape_reset_dist;
  config.escape_reset_theta = c->escape_reset_theta;
  config.vx_samples = c->vx_samples; config.vtheta_samples = c->vtheta_samples;
  config.heading_lookahead = c->heading_lookahead;
  config.holonomic_robot = c->holonomic_robot != 0;
  config.escape_vel = c->backup_vel;
  config.dwa = c->dwa != 0;
  config.heading_scoring = c->heading_scoring != 0;
  config.heading_scoring_timestep = c->heading_scoring_timestep;
  config.simple_attractor = c->simple_attractor != 0;
  std::string y;  // parsed back by reconfigure; %.17g round-trips every double
  for (int i = 0; i < c->n_y_vels; ++i) {
    char buf[32];
    snprintf(buf, sizeof(buf), "%s%.17g", i ? "," : "", c->y_vels[i]);
    y += buf;
  }
  config.y_vels = y;
  h->tp->sim_period_ = c->sim_period;  // a construction parameter (trajectory_planner.cpp:135-187) navo_tp_config carries
  h->tp->reconfigure(config);
}
void navo_tp_set_footprint(void* hv, const double* xy, int n) {
  static_cast<TpHandle*>(hv)->tp->setFootprint(toPoints(xy, n));
}
void navo_tp_set_costmap(void* hv, const uint8_t* grid, double ox, double oy) {
  setCostmap(static_cast<TpHandle*>(hv)->costmap, grid, ox, oy);
}
void navo_tp_update_plan(void* hv, const double* plan_xy, int n) {
  static_cast<TpHandle*>(hv)->tp->updatePlan(toPoses(plan_xy, n), false);
}

int navo_tp_find_best_path(void* hv, const double pose[3], const double vel[3], navo_tp_result* result, double* points,
                           int points_capacity) {
  TpHandle* h = static_cast<TpHandle*>(hv);
  tf::Stamped<tf::Pose> gp, gv, drive;
  gp.origin = tf::Vector3(pose[0], pose[1], 0.0); gp.yaw = pose[2];
  gv.origin = tf::Vector3(vel[0], vel[1], 0.0); gv.yaw = vel[2];
  Trajectory best = h->tp->findBestPath(gp, gv, drive);
  result->cost = best.cost_; result->xv = best.xv_; result->yv = best.yv_; result->thetav = best.thetav_;
  result->n_points = (int)best.getPointsSize();
  const TrajectoryPlanner& t = *h->tp;
  result->flags = (t.stuck_left ? 1 : 0) | (t.stuck_right ? 2 : 0) | (t.stuck_left_strafe ? 4 : 0) |
                  (t.stuck_right_strafe ? 8 : 0) | (t.rotating_left ? 16 : 0) | (t.rotating_right ? 32 : 0) |
                  (t.strafe_left ? 64 : 0) | (t.strafe_right ? 128 : 0) | (t.escaping_ ? 256 : 0);
  for (int i = 0; i < result->n_points && i < points_capacity; ++i)
    best.getPoint(i, points[3 * i], points[3 * i + 1], points[3 * i + 2]);
  return 0;
}

double navo_tp_score_trajectory(void* hv, const double pose[3], const double vel[3], const double vs[3]) {
  return static_cast<TpHandle*>(hv)->tp->scoreTrajectory(pose[0], pose[1], pose[2], vel[0], vel[1], vel[2], vs[0],
                                                         vs[1], vs[2]);
}

void navo_tp_get_grid(void* hv, int which, double* out) {
  TpHandle* h = static_cast<TpHandle*>(hv);
  MapGrid& g = which == 0 ? h->tp->path_map_ : h->tp->goal_map_;
  for (unsigned y = 0; y < g.size_y_; ++y)
    for (unsigned x = 0; x < g.size_x_; ++x) out[size_t(y) * g.size_x_ + x] = g(x, y).target_dist;
}

}  // extern "C"
