// Shared between the prefilter (voxelgrid.cu) and the NDT target voxelisation (ndt.cu):
// crop + bbox + key + radix sort + segment heads, i.e. "which points fall in which voxel, in index order".
#pragma once
#include "common.cuh"

namespace lgs {

struct CropParams {
  double range_min;  // < 0: disabled
  double box[6];
  int use_box;
};

struct GridParams {
  float inv[3];
  int min_b[3];
  int mul[3];
  unsigned sentinel;  // key given to cropped points: sorts after every real voxel
};

// The same grid with a 64-bit linear index (the wide VoxelGrid, used beyond INT32_MAX cells)
struct GridParamsWide {
  float inv[3];
  int min_b[3];
  unsigned long long mul[3];
  unsigned long long sentinel;  // larger than every real index
};

// Result of the shared front half.  Pointers live in ctx->tmp[] arenas and stay valid until the next
// call that uses the same context.
struct SortedVoxels {
  int status = 0;            // LGS_VG_OK / LGS_VG_REFUSED_OVERFLOW
  int64_t n_kept = 0;        // points surviving the crop (sorted entries [0, n_kept) are real)
  int n_seg = 0;             // occupied voxels
  const unsigned* keys = nullptr;   // sorted voxel indices (n entries, cropped ones at the tail); null for 64-bit keys
  const unsigned* vals = nullptr;   // point index of each sorted entry
  const int* seg_start = nullptr;   // n_seg offsets into keys/vals
  const unsigned char* keep = nullptr;
  int min_b[3] = {0, 0, 0}, max_b[3] = {0, 0, 0}, div_b[3] = {0, 0, 0};
  uint64_t total_cells = 0;
};

// wide: the wide VoxelGrid.  Where the narrow grid does not refuse it runs the narrow code; beyond that the index is 64
// bits wide and the refusal moves to the limits of int64 (DESIGN section 11).  The per-point index then goes to
// voxel_idx64_dev (voxel_idx_dev must be null).
int build_sorted_voxels(lgs_ctx* ctx, const float4* pts, int64_t n, const float leaf[3], double range_min, const double* box6,
                        int* voxel_idx_dev, int* member_rank_dev, SortedVoxels* out, bool wide = false, int64_t* voxel_idx64_dev = nullptr);

// Prefilter core on device buffers (voxelgrid.cu); out_pts_dev needs capacity n.
int voxelgrid_device(lgs_ctx* ctx, const float4* pts, int64_t n, const float leaf[3], int min_pts, double range_min, const double* box6,
                     float4* out_pts_dev, int* voxel_idx_dev, int* member_rank_dev, lgs_voxelgrid_info* info, bool wide = false,
                     int64_t* voxel_idx64_dev = nullptr);

}  // namespace lgs
