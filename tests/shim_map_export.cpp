// Compile-and-link check of the map export in the C++ shim (include/lgs/registration.hpp): VoxelGrid::setWideIndices and
// KeyFrameArray::exportMap, the save_map call sequence (GBS:469-501).  Runs the calls only with --run (needs a GPU).
#include <cstdio>
#include <cstring>

#include "lgs/registration.hpp"

int main(int argc, char** argv) {
  if (!(argc > 1 && std::strcmp(argv[1], "--run") == 0)) {
    std::printf("shim compiled; version %s\n", lgs_version());
    return 0;
  }
  // two points 5 km apart at a 1 cm leaf: 5e5^3 cells, far beyond INT32_MAX
  auto cloud = std::make_shared<lgs::PointCloud>();
  cloud->push_back(lgs::PointXYZI{0.0f, 0.0f, 0.0f, 1.0f, 1.0f, 0, 0, 0});
  cloud->push_back(lgs::PointXYZI{5000.0f, 5000.0f, 5000.0f, 1.0f, 2.0f, 0, 0, 0});
  lgs::VoxelGrid narrow, wide;
  lgs::PointCloud out_narrow, out_wide;
  for (lgs::VoxelGrid* vg : {&narrow, &wide}) {
    vg->setLeafSize(0.01f, 0.01f, 0.01f);
    vg->setInputCloud(cloud);
  }
  wide.setWideIndices(true);
  narrow.filter(out_narrow);
  wide.filter(out_wide);
  if (!narrow.ok() || narrow.info().status != LGS_VG_REFUSED_OVERFLOW) return 1;
  if (!wide.ok() || wide.info().status != LGS_VG_OK || out_wide.size() != 2 || wide.wideVoxelIndices().size() != 2) return 2;
  if (wide.wideVoxelIndices()[0] != 0 || wide.wideVoxelIndices()[1] <= static_cast<int64_t>(INT32_MAX)) return 3;
  lgs::KeyFrameArray key_frames;
  lgs::Matrix4f pose = lgs::Identity4f();
  key_frames.push(*cloud, pose, 0.0);
  pose[12] = 1.0f;
  key_frames.push(*cloud, pose, 1.0);
  const float* map_dev = nullptr;
  int64_t n_map = 0;
  lgs_voxelgrid_info info{};
  if (!key_frames.exportMap({}, 0.01f, &map_dev, &n_map, &info) || n_map != 4 || info.status != LGS_VG_OK) return 4;
  if (!key_frames.exportMap({1}, 0.0f, &map_dev, &n_map) || n_map != 2) return 5;
  std::printf("map export: %lld points, wide index of the far point %lld\n", static_cast<long long>(n_map),
              static_cast<long long>(wide.wideVoxelIndices()[1]));
  return 0;
}
