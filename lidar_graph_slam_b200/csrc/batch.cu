// Batched loop-closure verification: GBS:297-322 (VoxelGrid 0.5 m on the submap, setInputTarget / setInputSource,
// align with identity guess, getFinalTransformation / getFitnessScore / hasConverged) for a list of candidate
// pairs.  Pairs are independent, so W host workers each drive their own stream and registration object and pull
// pairs from a shared counter; kernels of different pairs overlap on the device.  Every pair runs entirely on one
// stream with deterministic reductions, so a pair's record does not depend on W, on the pair order, or on which
// GPU of the box it was dealt to.
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <mutex>
#include <thread>
#include <vector>

#include "dist.cuh"
#include "gicp.cuh"
#include "keyframes.cuh"
#include "voxel_common.cuh"

using namespace lgs;

namespace {

struct BatchShared {
  const lgs_batch_params* bp;
  int device;
  int64_t n_pairs;
  const void* const* scans;
  const int64_t* n_scan;
  const void* const* submaps;
  const int64_t* n_submap;
  int32_t stride;
  const float* guesses;
  int32_t pair_id0;
  lgs_align_result* records;
  // key-frame mode (lgs_batch_align_keyframes): pair i = key frame scan_ids[i] against the neighbourhood of center_ids[i]
  const lgs_keyframes* kf = nullptr;
  const int32_t* scan_ids = nullptr;
  const int32_t* center_ids = nullptr;
  int32_t search_key_frame_num = 0;
  // record sinks: pair i's record goes to records[i] (host) and, when rec_dev is set, is also stored at rec_dev[i] by the
  // pair's last kernel (its getFitnessScore reduction): rec_dev is the NCCL send buffer of lgs_batch_align*_dist
  lgs_align_result* rec_dev = nullptr;
  const int32_t* pair_ids = nullptr;  // global ids of the local pairs (distributed batch); otherwise pair_id0 + i
  std::atomic<int64_t> next{0};
  std::atomic<int> failed{0};
  std::mutex err_mu;
  std::string err;
};

// development aid: LGS_BATCH_TRACE=1 prints the host wall time of every stage of every pair (with a stream
// synchronisation after each stage, so the numbers are not the production timeline)
struct StageClock {
  bool on;
  cudaStream_t st;
  std::chrono::steady_clock::time_point t0;
  double ms[6] = {0, 0, 0, 0, 0, 0};
  explicit StageClock(cudaStream_t s) : on(getenv("LGS_BATCH_TRACE") != nullptr), st(s) {
    if (on) t0 = std::chrono::steady_clock::now();
  }
  void lap(int k) {
    if (!on) return;
    cudaStreamSynchronize(st);
    const auto t1 = std::chrono::steady_clock::now();
    ms[k] = std::chrono::duration<double, std::milli>(t1 - t0).count();
    t0 = t1;
  }
};

int run_pair(lgs_ctx* ctx, lgs_gicp* gicp, lgs_ndt* ndt, lgs_icp* icp, lgs_gicp_omp* gomp, DevBuf* sub_raw, DevBuf* sub_ds, DevBuf* scan_buf, BatchShared* S, int64_t i) {
  const lgs_batch_params& bp = *S->bp;
  lgs_align_result& rec = S->records[i];
  memset(&rec, 0, sizeof(rec));
  StageClock clk(ctx->stream);
  // submap -> (optional) VoxelGrid -> device-resident target
  int64_t n_tgt = 0;
  const float* scan_dev = nullptr;  // key-frame mode: the scan is a device cloud as well
  int64_t n_scan_dev = 0;
  if (S->kf) {
    // GBS:297-309: key frames min_id - K .. min_id + K that exist, ascending; GBS:247-251: the scan in the map frame
    std::vector<int32_t> ids;
    const int64_t count = keyframes_count(S->kf);
    for (int32_t d = -S->search_key_frame_num; d <= S->search_key_frame_num; d++) {
      const int64_t id = static_cast<int64_t>(S->center_ids[i]) + d;
      if (id >= 0 && id < count) ids.push_back(static_cast<int32_t>(id));
    }
    LGS_TRY(keyframes_assemble_into(S->kf, ctx, ids.data(), static_cast<int32_t>(ids.size()), &ctx->tmp[2], sub_raw, &n_tgt));
  } else {
    LGS_TRY(upload_cloud(ctx, S->submaps[i], S->n_submap[i], S->stride, sub_raw));
    n_tgt = S->n_submap[i];
  }
  clk.lap(0);
  const float* tgt_dev = sub_raw->as<float>();
  if (bp.submap_leaf > 0 && n_tgt > 0) {
    LGS_TRY(sub_ds->reserve(static_cast<size_t>(n_tgt) * 16));
    const float leaf[3] = {bp.submap_leaf, bp.submap_leaf, bp.submap_leaf};
    lgs_voxelgrid_info info;
    LGS_TRY(voxelgrid_device(ctx, sub_raw->as<float4>(), n_tgt, leaf, 0, -1.0, nullptr, sub_ds->as<float4>(), nullptr, nullptr, &info));
    tgt_dev = sub_ds->as<float>();
    n_tgt = info.n_out;
  }
  clk.lap(1);
  if (S->kf) {
    // into the worker's own buffer: setInputTarget may voxelise at once and use every scratch arena of the context
    LGS_TRY(keyframes_assemble_into(S->kf, ctx, S->scan_ids + i, 1, &ctx->tmp[2], scan_buf, &n_scan_dev));
    scan_dev = scan_buf->as<float>();
  }
  const float* guess = S->guesses ? S->guesses + 16 * i : nullptr;
  const int32_t pair_id = S->pair_ids ? S->pair_ids[i] : S->pair_id0 + static_cast<int32_t>(i);
  // arms the one-shot record sink of this context: the fitness kernel that follows completes and stores the record
  auto arm_record = [&]() {
    rec.pair_id = pair_id;
    if (S->rec_dev) {
      ctx->rec_out_proto = rec;
      ctx->rec_out_dev = S->rec_dev + i;
    }
  };
  const double max_range = bp.fitness_max_range > 0 ? bp.fitness_max_range : std::numeric_limits<double>::max();
  if (bp.method == LGS_METHOD_GICP) {
    LGS_TRY(lgs_gicp_set_target_dev(gicp, tgt_dev, n_tgt));
    clk.lap(2);
    if (scan_dev)
      LGS_TRY(lgs_gicp_set_source_dev(gicp, scan_dev, n_scan_dev));
    else
      LGS_TRY(lgs_gicp_set_source(gicp, S->scans[i], S->n_scan[i], S->stride));
    clk.lap(3);
    LGS_TRY(lgs_gicp_align(gicp, guess, &rec, nullptr));
    clk.lap(4);
    arm_record();
    LGS_TRY(lgs_gicp_fitness(gicp, max_range, &rec.fitness));
    clk.lap(5);
  } else if (bp.method == LGS_METHOD_ICP) {
    LGS_TRY(lgs_icp_set_target_dev(icp, tgt_dev, n_tgt));
    clk.lap(2);
    if (scan_dev)
      LGS_TRY(lgs_icp_set_source_dev(icp, scan_dev, n_scan_dev));
    else
      LGS_TRY(lgs_icp_set_source(icp, S->scans[i], S->n_scan[i], S->stride));
    clk.lap(3);
    LGS_TRY(lgs_icp_reset_convergence_criteria(icp));  // every pair starts from a fresh criteria object (order independence)
    LGS_TRY(lgs_icp_align(icp, guess, &rec, nullptr));
    clk.lap(4);
    arm_record();
    LGS_TRY(lgs_icp_fitness(icp, max_range, &rec.fitness));
    clk.lap(5);
  } else if (bp.method == LGS_METHOD_GICP_OMP) {
    LGS_TRY(lgs_gicp_omp_set_target_dev(gomp, tgt_dev, n_tgt));
    clk.lap(2);
    if (scan_dev)
      LGS_TRY(lgs_gicp_omp_set_source_dev(gomp, scan_dev, n_scan_dev));
    else
      LGS_TRY(lgs_gicp_omp_set_source(gomp, S->scans[i], S->n_scan[i], S->stride));
    clk.lap(3);
    LGS_TRY(lgs_gicp_omp_align(gomp, guess, &rec, nullptr));
    clk.lap(4);
    arm_record();
    LGS_TRY(lgs_gicp_omp_fitness(gomp, max_range, &rec.fitness));
    clk.lap(5);
  } else {
    LGS_TRY(lgs_ndt_set_target_dev(ndt, tgt_dev, n_tgt));
    clk.lap(2);
    if (scan_dev)
      LGS_TRY(lgs_ndt_set_source_dev(ndt, scan_dev, n_scan_dev));
    else
      LGS_TRY(lgs_ndt_set_source(ndt, S->scans[i], S->n_scan[i], S->stride));
    clk.lap(3);
    LGS_TRY(lgs_ndt_align(ndt, guess, &rec, nullptr));
    clk.lap(4);
    arm_record();
    LGS_TRY(lgs_ndt_fitness(ndt, max_range, &rec.fitness));
    clk.lap(5);
  }
  if (clk.on)
    fprintf(stderr, "[lgs batch] pair %lld: upload %.2f  voxelgrid %.2f  set_target %.2f  set_source %.2f  align %.2f  fitness %.2f ms (target %lld pts)\n",
            static_cast<long long>(i), clk.ms[0], clk.ms[1], clk.ms[2], clk.ms[3], clk.ms[4], clk.ms[5], static_cast<long long>(n_tgt));
  rec.pair_id = pair_id;
  return LGS_OK;
}

// A worker's device state (stream, registration objects, staging buffers) outlives the call: creating a stream, the
// pinned result mailbox and ~20 device buffers costs tens of milliseconds, more than verifying a pair.  Slots live in
// a per-process pool keyed by device; lgs_batch_align borrows W of them and returns them; lgs_batch_release frees them.
struct WorkerSlot {
  int device = -1;
  lgs_ctx* ctx = nullptr;
  lgs_gicp* gicp = nullptr;
  lgs_ndt* ndt = nullptr;
  lgs_icp* icp = nullptr;
  lgs_gicp_omp* gomp = nullptr;
  DevBuf sub_raw, sub_ds, scan_buf;
  void destroy() {
    if (ctx) {
      cudaSetDevice(device);
      cudaStreamSynchronize(ctx->stream);
    }
    sub_raw.release();
    sub_ds.release();
    scan_buf.release();
    if (gicp) lgs_gicp_destroy(gicp);
    if (ndt) lgs_ndt_destroy(ndt);
    if (icp) lgs_icp_destroy(icp);
    if (gomp) lgs_gicp_omp_destroy(gomp);
    if (ctx) lgs_ctx_destroy(ctx);
    ctx = nullptr;
    gicp = nullptr;
    ndt = nullptr;
    icp = nullptr;
    gomp = nullptr;
  }
};

std::mutex g_pool_mu;
std::vector<WorkerSlot*> g_pool;  // idle slots

WorkerSlot* borrow_slot(int device) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  for (size_t i = 0; i < g_pool.size(); i++)
    if (g_pool[i]->device == device) {
      WorkerSlot* w = g_pool[i];
      g_pool.erase(g_pool.begin() + i);
      return w;
    }
  WorkerSlot* w = new WorkerSlot;
  w->device = device;
  return w;
}

void return_slot(WorkerSlot* w) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  g_pool.push_back(w);
}

void worker(BatchShared* S) {
  WorkerSlot* w = borrow_slot(S->device);
  int rc = LGS_OK;
  const lgs_batch_params& bp = *S->bp;
  if (!w->ctx) rc = lgs_ctx_create(S->device, nullptr, &w->ctx);
  if (rc == LGS_OK) w->ctx->polite_wait = true;
  if (rc == LGS_OK) rc = use_device(w->ctx);
  if (rc == LGS_OK) {
    if (bp.method == LGS_METHOD_GICP) {
      if (!w->gicp) rc = lgs_gicp_create(w->ctx, &w->gicp);
      if (rc == LGS_OK) {
        // every call starts from the library defaults (fast_gicp.hpp / gicp_settings.hpp), then the batch's settings
        lgs_gicp_set_correspondence_randomness(w->gicp, bp.k_correspondences > 0 ? bp.k_correspondences : 20);
        lgs_gicp_set_maximum_iterations(w->gicp, bp.max_iterations > 0 ? bp.max_iterations : 64);
        lgs_gicp_set_transformation_epsilon(w->gicp, bp.transformation_epsilon > 0 ? bp.transformation_epsilon : 5e-4);
        lgs_gicp_set_max_correspondence_distance(w->gicp, bp.max_correspondence_distance > 0 ? bp.max_correspondence_distance
                                                                                              : static_cast<double>(std::numeric_limits<float>::max()));
      }
    } else if (bp.method == LGS_METHOD_ICP) {
      if (!w->icp) rc = lgs_icp_create(w->ctx, &w->icp);
      if (rc == LGS_OK) {  // PCL defaults, then the batch's settings (GBS:145-148)
        lgs_icp_set_maximum_iterations(w->icp, bp.max_iterations > 0 ? bp.max_iterations : 10);
        lgs_icp_set_transformation_epsilon(w->icp, bp.transformation_epsilon > 0 ? bp.transformation_epsilon : 0.0);
        lgs_icp_set_max_correspondence_distance(w->icp, bp.max_correspondence_distance > 0 ? bp.max_correspondence_distance : 1.3407807929942596e154);
        lgs_icp_set_euclidean_fitness_epsilon(w->icp, bp.euclidean_fitness_epsilon != 0 ? bp.euclidean_fitness_epsilon : -std::numeric_limits<double>::max());
        lgs_icp_set_transformation_rotation_epsilon(w->icp, 0.0);
      }
    } else if (bp.method == LGS_METHOD_GICP_OMP) {
      if (!w->gomp) rc = lgs_gicp_omp_create(w->ctx, &w->gomp);
      if (rc == LGS_OK) {  // gicp_omp.h:116-126 defaults, then the batch's settings (GBS:134-137)
        lgs_gicp_omp_set_correspondence_randomness(w->gomp, bp.k_correspondences > 0 ? bp.k_correspondences : 20);
        lgs_gicp_omp_set_maximum_iterations(w->gomp, bp.max_iterations > 0 ? bp.max_iterations : 200);
        lgs_gicp_omp_set_transformation_epsilon(w->gomp, bp.transformation_epsilon > 0 ? bp.transformation_epsilon : 5e-4);
        lgs_gicp_omp_set_max_correspondence_distance(w->gomp, bp.max_correspondence_distance > 0 ? bp.max_correspondence_distance : 5.0);
        lgs_gicp_omp_set_maximum_optimizer_iterations(w->gomp, bp.max_optimizer_iterations > 0 ? bp.max_optimizer_iterations : 20);
      }
    } else {
      if (!w->ndt) rc = lgs_ndt_create(w->ctx, &w->ndt);
      if (rc == LGS_OK) {
        lgs_ndt_set_resolution(w->ndt, bp.ndt_resolution > 0 ? bp.ndt_resolution : 1.0f);
        lgs_ndt_set_step_size(w->ndt, bp.ndt_step_size > 0 ? bp.ndt_step_size : 0.1);
        lgs_ndt_set_maximum_iterations(w->ndt, bp.max_iterations > 0 ? bp.max_iterations : 35);
        lgs_ndt_set_transformation_epsilon(w->ndt, bp.transformation_epsilon > 0 ? bp.transformation_epsilon : 0.1);
      }
    }
  }
  while (rc == LGS_OK && !S->failed.load()) {
    const int64_t i = S->next.fetch_add(1);
    if (i >= S->n_pairs) break;
    rc = run_pair(w->ctx, w->gicp, w->ndt, w->icp, w->gomp, &w->sub_raw, &w->sub_ds, &w->scan_buf, S, i);
  }
  if (rc != LGS_OK) {
    std::lock_guard<std::mutex> lk(S->err_mu);
    if (!S->failed.exchange(rc)) S->err = lgs_last_error();
  }
  if (w->ctx) {
    cudaSetDevice(S->device);
    cudaStreamSynchronize(w->ctx->stream);
  }
  if (rc != LGS_OK) {  // a failed slot is not reused
    w->destroy();
    delete w;
  } else {
    return_slot(w);
  }
}

}  // namespace

static int run_batch(BatchShared& S);

extern "C" int lgs_batch_align(int device, void* cuda_stream, const lgs_batch_params* params, int64_t n_pairs, const void* const* scans,
                               const int64_t* n_scan, const void* const* submaps, const int64_t* n_submap, int32_t stride_bytes,
                               const float* guesses16, int32_t pair_id0, lgs_align_result* records, void* records_dev) {
  LGS_NVTX("lgs_batch_align");
  LGS_REQUIRE(params && records, "null argument");
  LGS_REQUIRE(n_pairs >= 0, "negative pair count");
  LGS_REQUIRE(params->method >= LGS_METHOD_NDT && params->method <= LGS_METHOD_GICP_OMP, "unknown method");
  LGS_REQUIRE(n_pairs == 0 || (scans && n_scan && submaps && n_submap), "null pair arrays");
  BatchShared S;
  S.bp = params;
  S.device = device;
  S.n_pairs = n_pairs;
  S.scans = scans;
  S.n_scan = n_scan;
  S.submaps = submaps;
  S.n_submap = n_submap;
  S.stride = stride_bytes;
  S.guesses = guesses16;
  S.pair_id0 = pair_id0;
  S.records = records;
  S.rec_dev = static_cast<lgs_align_result*>(records_dev);
  (void)cuda_stream;  // every worker synchronises its own stream before the call returns: records_dev is complete
  return run_batch(S);
}

// The same verification with both clouds of every pair taken from the device-resident key-frame array: pair i aligns key
// frame scan_ids[i] (in the map frame, GBS:247-251) to the VoxelGrid-filtered neighbourhood center_ids[i] +- search_key_frame_num
// (GBS:297-313).  Nothing but the 96-byte records crosses PCIe.
extern "C" int lgs_batch_align_keyframes(lgs_keyframes* kf, void* cuda_stream, const lgs_batch_params* params, int64_t n_pairs,
                                         const int32_t* scan_ids, const int32_t* center_ids, int32_t search_key_frame_num,
                                         const float* guesses16, int32_t pair_id0, lgs_align_result* records, void* records_dev) {
  LGS_NVTX("lgs_batch_align_keyframes");
  LGS_REQUIRE(kf && params && records, "null argument");
  LGS_REQUIRE(n_pairs >= 0 && search_key_frame_num >= 0, "negative count");
  LGS_REQUIRE(params->method >= LGS_METHOD_NDT && params->method <= LGS_METHOD_GICP_OMP, "unknown method");
  LGS_REQUIRE(n_pairs == 0 || (scan_ids && center_ids), "null pair arrays");
  const int64_t count = keyframes_count(kf);
  for (int64_t i = 0; i < n_pairs; i++)
    LGS_REQUIRE(scan_ids[i] >= 0 && scan_ids[i] < count && center_ids[i] >= 0 && center_ids[i] < count, "key frame id out of range");
  LGS_TRY(keyframes_wait_resident(kf));
  BatchShared S;
  S.bp = params;
  S.device = keyframes_device(kf);
  S.n_pairs = n_pairs;
  S.scans = nullptr;
  S.n_scan = nullptr;
  S.submaps = nullptr;
  S.n_submap = nullptr;
  S.stride = 16;
  S.guesses = guesses16;
  S.pair_id0 = pair_id0;
  S.records = records;
  S.kf = kf;
  S.scan_ids = scan_ids;
  S.center_ids = center_ids;
  S.search_key_frame_num = search_key_frame_num;
  S.rec_dev = static_cast<lgs_align_result*>(records_dev);
  (void)cuda_stream;
  return run_batch(S);
}

static int run_batch(BatchShared& S) {
  const lgs_batch_params* params = S.bp;
  const int64_t n_pairs = S.n_pairs;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    set_error("no CUDA device available; this library has no CPU fallback");
    return LGS_ERR_CUDA;
  }
  int W = params->n_workers > 0 ? params->n_workers : 8;  // measured on one B200: 2 276 / 2 726 / 2 609 pairs/s at 4 / 8 / 12 workers
  if (W > n_pairs) W = static_cast<int>(std::max<int64_t>(n_pairs, 1));
  if (W > 32) W = 32;
  std::vector<std::thread> threads;
  for (int w = 0; w < W; w++) threads.emplace_back(worker, &S);
  for (auto& t : threads) t.join();
  if (S.failed.load()) {
    set_error("lgs_batch_align: %s", S.err.c_str());
    return S.failed.load();
  }
  return LGS_OK;
}

// ---- the batch over the GPUs of a box (SURVEY section 8e) -----------------------------------------------------------
namespace {

// partition -> local verification with the send buffer as record sink -> one ncclAllGather -> records_all[pair id]
template <typename FillLocal>
int run_dist(lgs_comm* comm, int device, const int64_t* sizes, int64_t n_pairs, lgs_align_result* records_all, lgs_batch_dist_info* info, BatchShared& S,
             FillLocal fill_local) {
  if (device != comm->device) {
    set_error("the communicator lives on device %d, the batch on device %d", comm->device, device);
    return LGS_ERR_INVALID;
  }
  LGS_CUDA(cudaSetDevice(device));
  std::vector<int32_t> mine;
  partition_pairs(sizes, n_pairs, comm->rank, comm->world, &mine);
  const int64_t cap = std::max<int64_t>(1, (n_pairs + comm->world - 1) / comm->world);
  LGS_TRY(comm->send.reserve(static_cast<size_t>(cap) * sizeof(lgs_align_result)));
  cudaStream_t st = nullptr;  // the gather runs on the legacy default stream: it orders after the memset below and,
                              // because every worker synchronises its own stream before returning, after the records
  LGS_CUDA(cudaMemsetAsync(comm->send.p, 0xFF, static_cast<size_t>(cap) * sizeof(lgs_align_result), st));  // pair_id = -1: unused slot
  LGS_CUDA(cudaStreamSynchronize(st));
  std::vector<lgs_align_result> local(mine.size());
  S.n_pairs = static_cast<int64_t>(mine.size());
  S.records = local.data();
  S.rec_dev = comm->send.as<lgs_align_result>();
  S.pair_ids = mine.data();
  S.pair_id0 = 0;
  S.device = device;
  fill_local(mine);
  const auto t0 = std::chrono::steady_clock::now();
  LGS_TRY(run_batch(S));
  const auto t1 = std::chrono::steady_clock::now();
  int64_t got = 0;
  LGS_TRY(comm_all_gather(comm, st, cap, sizeof(lgs_align_result), [&](const void* p) {
    const lgs_align_result* r = static_cast<const lgs_align_result*>(p);
    if (r->pair_id < 0) return 0;  // unused slot of a rank with fewer pairs
    if (r->pair_id >= n_pairs) {
      set_error("gathered record carries pair id %d outside [0, %lld)", r->pair_id, static_cast<long long>(n_pairs));
      return LGS_ERR_STATE;
    }
    records_all[r->pair_id] = *r;
    return 1;
  }, &got));
  const auto t2 = std::chrono::steady_clock::now();
  if (info) {
    info->rank = comm->rank;
    info->world = comm->world;
    info->n_local = static_cast<int64_t>(mine.size());
    info->n_received = got;
    info->gather_bytes = cap * comm->world * static_cast<int64_t>(sizeof(lgs_align_result));
    info->verify_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    info->gather_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
  }
  if (got != n_pairs) {
    set_error("the gather returned %lld of %lld records", static_cast<long long>(got), static_cast<long long>(n_pairs));
    return LGS_ERR_STATE;
  }
  return LGS_OK;
}

}  // namespace

extern "C" int lgs_batch_align_keyframes_dist(lgs_keyframes* kf, lgs_comm* comm, const lgs_batch_params* params, int64_t n_pairs,
                                              const int32_t* scan_ids, const int32_t* center_ids, int32_t search_key_frame_num,
                                              const float* guesses16, lgs_align_result* records_all, lgs_batch_dist_info* info) {
  LGS_NVTX("lgs_batch_align_keyframes_dist");
  LGS_REQUIRE(kf && comm && params && (records_all || n_pairs == 0), "null argument");
  LGS_REQUIRE(n_pairs >= 0 && n_pairs < (int64_t(1) << 31) && search_key_frame_num >= 0, "count out of range");
  LGS_REQUIRE(params->method >= LGS_METHOD_NDT && params->method <= LGS_METHOD_GICP_OMP, "unknown method");
  LGS_REQUIRE(n_pairs == 0 || (scan_ids && center_ids), "null pair arrays");
  const int64_t count = keyframes_count(kf);
  std::vector<int64_t> sizes(static_cast<size_t>(n_pairs));
  for (int64_t i = 0; i < n_pairs; i++) {
    LGS_REQUIRE(scan_ids[i] >= 0 && scan_ids[i] < count && center_ids[i] >= 0 && center_ids[i] < count, "key frame id out of range");
    int64_t sz = keyframes_points(kf, scan_ids[i]);
    for (int64_t id = std::max<int64_t>(0, static_cast<int64_t>(center_ids[i]) - search_key_frame_num);
         id <= std::min<int64_t>(count - 1, static_cast<int64_t>(center_ids[i]) + search_key_frame_num); id++)
      sz += keyframes_points(kf, id);
    sizes[static_cast<size_t>(i)] = sz;
  }
  LGS_TRY(keyframes_wait_resident(kf));
  BatchShared S;
  S.bp = params;
  S.scans = nullptr;
  S.n_scan = nullptr;
  S.submaps = nullptr;
  S.n_submap = nullptr;
  S.stride = 16;
  S.kf = kf;
  S.search_key_frame_num = search_key_frame_num;
  std::vector<int32_t> sid, cid;
  std::vector<float> gl;
  return run_dist(comm, keyframes_device(kf), sizes.data(), n_pairs, records_all, info, S, [&](const std::vector<int32_t>& mine) {
    for (int32_t i : mine) {
      sid.push_back(scan_ids[i]);
      cid.push_back(center_ids[i]);
      if (guesses16) gl.insert(gl.end(), guesses16 + 16 * static_cast<size_t>(i), guesses16 + 16 * static_cast<size_t>(i) + 16);
    }
    S.scan_ids = sid.data();
    S.center_ids = cid.data();
    S.guesses = guesses16 ? gl.data() : nullptr;
  });
}

extern "C" int lgs_batch_align_dist(lgs_comm* comm, const lgs_batch_params* params, int64_t n_pairs, const void* const* scans, const int64_t* n_scan,
                                    const void* const* submaps, const int64_t* n_submap, int32_t stride_bytes, const float* guesses16,
                                    lgs_align_result* records_all, lgs_batch_dist_info* info) {
  LGS_NVTX("lgs_batch_align_dist");
  LGS_REQUIRE(comm && params && (records_all || n_pairs == 0), "null argument");
  LGS_REQUIRE(n_pairs >= 0 && n_pairs < (int64_t(1) << 31), "count out of range");
  LGS_REQUIRE(params->method >= LGS_METHOD_NDT && params->method <= LGS_METHOD_GICP_OMP, "unknown method");
  LGS_REQUIRE(n_pairs == 0 || (scans && n_scan && submaps && n_submap), "null pair arrays");
  std::vector<int64_t> sizes(static_cast<size_t>(n_pairs));
  for (int64_t i = 0; i < n_pairs; i++) sizes[static_cast<size_t>(i)] = n_scan[i] + n_submap[i];
  BatchShared S;
  S.bp = params;
  S.stride = stride_bytes;
  std::vector<const void*> ls, lm;
  std::vector<int64_t> lns, lnm;
  std::vector<float> gl;
  return run_dist(comm, comm->device, sizes.data(), n_pairs, records_all, info, S, [&](const std::vector<int32_t>& mine) {
    for (int32_t i : mine) {
      ls.push_back(scans[i]);
      lm.push_back(submaps[i]);
      lns.push_back(n_scan[i]);
      lnm.push_back(n_submap[i]);
      if (guesses16) gl.insert(gl.end(), guesses16 + 16 * static_cast<size_t>(i), guesses16 + 16 * static_cast<size_t>(i) + 16);
    }
    S.scans = ls.data();
    S.n_scan = lns.data();
    S.submaps = lm.data();
    S.n_submap = lnm.data();
    S.guesses = guesses16 ? gl.data() : nullptr;
  });
}

extern "C" void lgs_batch_release(void) {
  std::vector<WorkerSlot*> all;
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    all.swap(g_pool);
  }
  for (WorkerSlot* w : all) {
    w->destroy();
    delete w;
  }
}
