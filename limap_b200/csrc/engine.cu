// engine.cu — host side of the C ABI declared in include/limap_b200.h: context, scene upload, batched
// TriangulateImage, result getters, ComputeLineTracks, line BA, VP detection, track filters and remerge.
//
// Mirrors (file:line under /root/reference/src/limap/):
//   BaseLineTriangulator::{Init,TriangulateImage,TriangulateImageExhaustiveMatch}
//       triangulation/base_line_triangulator.cc:45-136
//   GlobalLineTriangulator::{ScoringCallback,run_clustering,build_tracks_from_clusters,ComputeLineTracks}
//       triangulation/global_line_triangulator.cc:59-69, 234-359
//   merging::ComputeLineTrackLabelsGreedy      merging/merging.cc:18-103
//   merging::Aggregator::aggregate_line3d_list merging/aggregator.cc:53-101
// There is no CPU fallback: without a CUDA device lm_ctx_create fails with LM_ERR_NOGPU.
#include "../../include/limap_b200.h"
#include "tri_kernels.cuh"
#include "graph_kernels.cuh"
#include "lm_kernels.cuh"
#include "vp_kernels.cuh"
#include "merge_kernels.cuh"
#include "sfm_kernels.cuh"
#include <cub/device/device_run_length_encode.cuh>
#include <algorithm>
#include <chrono>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <map>
#include <queue>
#include <set>
#include <string>
#include <unordered_map>
#include <vector>

static_assert(sizeof(lm_node_record) == sizeof(lm::NodeRecord), "record layout");

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}
#define CU(call)                                                                                                    \
  do {                                                                                                              \
    cudaError_t e_ = (call);                                                                                        \
    if (e_ != cudaSuccess)                                                                                          \
      return fail(LM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                                 \
  } while (0)

namespace {

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct MatchBlock {
  int src_view, ng_view;
  int64_t n_rows;
  int64_t pair_off; // row offset into the device pairs store (-1: exhaustive)
  int order;        // insertion order within the source image (exhaustive mode keeps the given order)
};

struct M3h {
  double m[9];
};
static M3h quat_to_R(const double q_in[4]) { // base/pose.cc:12-18 (Eigen toRotationMatrix)
  double n = std::sqrt(q_in[0] * q_in[0] + q_in[1] * q_in[1] + q_in[2] * q_in[2] + q_in[3] * q_in[3]);
  double q[4];
  if (n == 0) { q[0] = 1; q[1] = q_in[1]; q[2] = q_in[2]; q[3] = q_in[3]; }
  else for (int i = 0; i < 4; ++i) q[i] = q_in[i] / n;
  const double w = q[0], x = q[1], y = q[2], z = q[3];
  const double tx = 2 * x, ty = 2 * y, tz = 2 * z, twx = tx * w, twy = ty * w, twz = tz * w;
  const double txx = tx * x, txy = ty * x, txz = tz * x, tyy = ty * y, tyz = tz * y, tzz = tz * z;
  M3h R;
  R.m[0] = 1 - (tyy + tzz); R.m[1] = txy - twz; R.m[2] = txz + twy;
  R.m[3] = txy + twz; R.m[4] = 1 - (txx + tzz); R.m[5] = tyz - twx;
  R.m[6] = txz - twy; R.m[7] = tyz + twx; R.m[8] = 1 - (txx + tyy);
  return R;
}

template <typename T> lm::LinkerDev<T> to_dev(const lm_linker_config &c) {
  lm::LinkerDev<T> d;
  d.score_th = (T)c.score_th; d.th_angle = (T)c.th_angle; d.th_overlap = (T)c.th_overlap;
  d.th_smartoverlap = (T)c.th_smartoverlap; d.th_smartangle = (T)c.th_smartangle; d.th_perp = (T)c.th_perp;
  d.th_innerseg = (T)c.th_innerseg; d.th_scaleinv = (T)c.th_scaleinv;
  d.mult = (T)(1.0 / std::sqrt(-std::log(c.score_th) * 2.0)); // line_linker.cc:9-13
  d.use_angle = c.use_angle; d.use_overlap = c.use_overlap; d.use_smartangle = c.use_smartangle;
  d.use_perp = c.use_perp; d.use_innerseg = c.use_innerseg; d.use_scaleinv = c.use_scaleinv;
  return d;
}

struct Track {
  std::vector<int> img, line, node;
  std::vector<int64_t> gid;
  double agg[7];
};

} // namespace

struct lm_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr;
  // match uploads run on their own stream so that a run can start on the first source images while the rest
  // of the tables is still crossing PCIe
  cudaStream_t copy_stream = nullptr;
  cudaStream_t prep_stream = nullptr; // row expansion + sort of pipeline group g+1 run under the node kernel of group g
  std::vector<cudaEvent_t> evp;       // per pipeline group: rows of the group sorted, node offsets known
  cudaEvent_t ev_run_begin = nullptr;
  cudaStream_t out_stream = nullptr;  // device -> host copies of finished groups (lm_tri_set_node_sink)
  char *node_sink = nullptr;
  DevBuf d_scan_tmp, d_local_off;
  struct CopyChunk { int64_t row_end; cudaEvent_t ev; };
  std::vector<CopyChunk> chunks;
  std::vector<cudaEvent_t> event_pool;
  double node_kernel_ms_acc = 0;
  DevBuf d_raw_blocks, d_bkey, d_bkey2, d_bval, d_bval2, d_blk_rows; // device mirror of `blocks` + sort scratch
  int64_t raw_uploaded = 0;
  cudaEvent_t ev_raw = nullptr; // recorded on the copy stream after the latest descriptor upload
  // Every host->device transfer (scene, VPs, matches) travels on the copy stream; the compute stream only waits
  // for events. A compute stream whose latest operation is itself a host->device copy has its next operations
  // (event records, kernel launches) ordered behind whatever the H2D copy engine is working on -- i.e. behind a
  // bulk match upload issued in between (measured in round 1: ~3 ms per hypersim100 step).
  cudaEvent_t ev_scene = nullptr;
  std::vector<lm::ViewD> h_views;    // staging of the scene tables (kept alive: the copies are asynchronous)
  std::vector<cudaEvent_t> evk;      // per pipeline group: node-kernel begin/end (read after the run's only sync)
  DevBuf d_gather;                   // [0] total edges, [1] overflow flag of the last unpack; +64: rank node table
  int64_t gather_tab[64] = {0};
  int gather_world = 0;
  bool edges_count_on_device = false; // n_edges_dev is still on the device (lm_tri_unpack_messages)
  int cap_hint = 0;                  // staging capacity of the node kernel, from the previous run (0: default)
  int cap_hint_cand = 0;             // the same for the split scorer: largest candidate count of a node (0: unknown)
  bool outside_shard_clean = false;  // node records / row offsets outside the shard were zero-filled
  int run_retry = 0;
  int sm_count = 148;
  int max_smem_optin = 0;
  // scene
  bool have_scene = false;
  int V = 0;
  std::vector<int> img_ids;
  std::unordered_map<int, int> id2view;
  std::vector<int64_t> line_off;
  int64_t n_nodes = 0;
  DevBuf d_views, d_segs, d_segs_raw, d_node_view, d_line_off, d_img_ids, d_host_edges;
  // config
  bool have_cfg = false;
  lm_tri_config cfg;
  bool ranges_flag = false;
  double rlo[3] = {0, 0, 0}, rhi[3] = {0, 0, 0};
  // InitVPResults
  bool have_vps = false;
  DevBuf d_vp_label, d_vp_voff, d_vp_vps;
  int ns = 1; // proposal slots per match row of the last run (3 with VP proposals)
  // staged matches
  std::vector<MatchBlock> blocks;
  std::vector<char> image_added;
  std::vector<int> image_norder;
  DevBuf d_pairs;
  int64_t pairs_rows = 0;
  bool any_exhaustive = false, any_matches = false;
  int shard_begin = 0, shard_end = -1;
  int pipeline_groups = 1; // lm_tri_set_pipeline_groups
  // pinned landing pad of the small device->host reads inside a run (no staging through pageable memory)
  unsigned int *h_pin = nullptr;
  // run buffers
  DevBuf d_blk_row_off, d_blk_src, d_blk_ng, d_blk_pair_off;
  DevBuf d_key, d_key2, d_val, d_val2, d_sort_tmp; // d_key / d_val: unsorted rows of the radix-sort path only
  DevBuf d_rs_vrow, d_rs_vtile, d_rs_vtab, d_rs_tab;  // counting-sort row preparation: per-view tables, tile table
  DevBuf d_node_row_off, d_scalars; // scalars: [0] max_rows(uint) [1] err(int) ; counters at +16
  DevBuf d_nodes, d_row_state, d_row_cand, d_slab, d_cand;
  DevBuf d_edges, d_edges2, d_edge_keys, d_edge_keys2, d_edge_w, d_edge_cnt;
  DevBuf d_g_flag, d_g_pos, d_g_kc, d_g_wc, d_g_occ, d_g_occ2, d_g_hk, d_g_hk2, d_g_gidx, d_g_gnode, d_g_k1, d_g_k1b, d_g_k2, d_g_k2b;
  DevBuf d_nvalid, d_edge_off, d_edge_ng; // compact valid_edges_ of the shard (node-major, candidate order)
  uint32_t *sorted_val = nullptr;
  uint32_t *sorted_key = nullptr;
  int64_t n_rows = 0;
  int64_t node_begin = 0, node_end = 0;
  bool ran = false;
  lm_tri_stats stats;
  // host caches (filled lazily after a run)
  bool h_nodes_valid = false;
  std::vector<lm::NodeRecord> h_nodes;
  bool h_rows_valid = false;
  std::vector<uint32_t> h_node_row_off, h_row_ng;
  std::vector<uint8_t> h_row_state;
  std::vector<double> h_row_cand;
  bool h_edges_valid = false;
  std::vector<uint32_t> h_edge_off, h_edge_ng;
  int64_t n_edges_dev = 0; // directed valid edges collected on device
  bool edges_collected = false;
  // line BA
  DevBuf d_ba_in, d_ba_blocks, d_ba_out;
  DevBuf d_vp_pts, d_vp_off, d_vp_labels, d_vp_nc, d_vp_ps, d_vp_mat;
  lm_ba_stats ba_stats;
  void *h_ba_pin = nullptr; // pinned landing pad of lm_ba_solve's results
  size_t h_ba_pin_cap = 0;
  lm_vp_stats vp_stats;
  DevBuf d_vp_idx;
  // track filters / remerge
  DevBuf d_mg_in, d_mg_out, d_mg_edges;
  DevBuf d_sfm_in, d_sfm_keys, d_sfm_keys2, d_sfm_a, d_sfm_b, d_sfm_c, d_sfm_d; // neighbour ranking scratch
  lm_merge_stats mg_stats;
  // tracks
  std::vector<Track> tracks;
  std::vector<std::pair<int, int>> graph_nodes;
};

namespace {

int sync_stream(lm_ctx *c) {
  CU(cudaStreamSynchronize(c->stream));
  return LM_OK;
}

int fetch_nodes(lm_ctx *c) {
  if (c->h_nodes_valid) return LM_OK;
  c->h_nodes.resize(c->n_nodes);
  CU(cudaMemcpyAsync(c->h_nodes.data(), c->d_nodes.p, sizeof(lm::NodeRecord) * c->n_nodes, cudaMemcpyDeviceToHost,
                     c->stream));
  CU(cudaStreamSynchronize(c->stream));
  c->h_nodes_valid = true;
  return LM_OK;
}
int fetch_rows(lm_ctx *c) {
  if (c->h_rows_valid) return LM_OK;
  c->h_node_row_off.resize(c->n_nodes + 1);
  c->h_row_ng.resize(c->n_rows);
  c->h_row_state.resize(c->n_rows * c->ns);
  CU(cudaMemcpyAsync(c->h_node_row_off.data(), c->d_node_row_off.p, 4 * (c->n_nodes + 1), cudaMemcpyDeviceToHost,
                     c->stream));
  if (c->n_rows) {
    CU(cudaMemcpyAsync(c->h_row_ng.data(), c->sorted_val, 4 * c->n_rows, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(c->h_row_state.data(), c->d_row_state.p, c->n_rows * c->ns, cudaMemcpyDeviceToHost, c->stream));
    if (c->cfg.debug_mode) {
      c->h_row_cand.resize(c->n_rows * c->ns * 10);
      CU(cudaMemcpyAsync(c->h_row_cand.data(), c->d_row_cand.p, 80 * c->n_rows * c->ns, cudaMemcpyDeviceToHost, c->stream));
    }
  }
  CU(cudaStreamSynchronize(c->stream));
  c->h_rows_valid = true;
  return LM_OK;
}

int fetch_edges(lm_ctx *c) {
  if (c->h_edges_valid) return LM_OK;
  const int64_t n = c->node_end - c->node_begin;
  c->h_edge_off.assign(n + 1, 0);
  c->h_edge_ng.resize(c->stats.n_valid_edges);
  if (n > 0) {
    CU(cudaMemcpyAsync(c->h_edge_off.data(), c->d_edge_off.p, 4 * (n + 1), cudaMemcpyDeviceToHost, c->stream));
    if (c->stats.n_valid_edges)
      CU(cudaMemcpyAsync(c->h_edge_ng.data(), c->d_edge_ng.p, 4 * c->stats.n_valid_edges, cudaMemcpyDeviceToHost,
                         c->stream));
  }
  CU(cudaStreamSynchronize(c->stream));
  c->h_edges_valid = true;
  return LM_OK;
}

int ensure_ran(lm_ctx *c) {
  if (c->ran) return LM_OK;
  return lm_tri_run(c);
}

} // namespace

extern "C" {

const char *lm_last_error(void) { return g_err.c_str(); }
const char *lm_version(void) { return "limap_b200 0.1 (sm_100a)"; }

int lm_ctx_create(int device, lm_ctx **out) {
  if (!out) return fail(LM_ERR_INVALID, "out is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(LM_ERR_NOGPU, std::string("no CUDA device (") + cudaGetErrorString(e) +
                                  "); limap_b200 has no CPU fallback");
  if (device < 0 || device >= n) return fail(LM_ERR_INVALID, "device index out of range");
  CU(cudaSetDevice(device));
  lm_ctx *c = new lm_ctx();
  c->device = device;
  CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->own_stream = true;
  CU(cudaEventCreate(&c->ev0));
  CU(cudaEventCreate(&c->ev1));
  CU(cudaEventCreate(&c->evk0));
  CU(cudaEventCreate(&c->evk1));
  CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  {
    int lo_p = 0, hi_p = 0; // (numerically lowest = greatest priority: the small preparation kernels take the next free SM slots)
    CU(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
    CU(cudaStreamCreateWithPriority(&c->prep_stream, cudaStreamNonBlocking, hi_p));
    CU(cudaStreamCreateWithPriority(&c->out_stream, cudaStreamNonBlocking, hi_p));
    CU(cudaEventCreateWithFlags(&c->ev_run_begin, cudaEventDisableTiming));
  }
  CU(cudaHostAlloc(reinterpret_cast<void **>(&c->h_pin), 2048, cudaHostAllocDefault));
  CU(cudaEventCreateWithFlags(&c->ev_scene, cudaEventDisableTiming));
  cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
  cudaDeviceGetAttribute(&c->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  memset(&c->stats, 0, sizeof(c->stats));
  memset(&c->ba_stats, 0, sizeof(c->ba_stats));
  memset(&c->vp_stats, 0, sizeof(c->vp_stats));
  memset(&c->mg_stats, 0, sizeof(c->mg_stats));
  *out = c;
  return LM_OK;
}

void lm_ctx_destroy(lm_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  DevBuf *bufs[] = {&c->d_scan_tmp, &c->d_local_off, &c->d_segs_raw, &c->d_img_ids, &c->d_host_edges, &c->d_views, &c->d_segs, &c->d_node_view, &c->d_line_off, &c->d_pairs, &c->d_blk_row_off,
                    &c->d_blk_src, &c->d_blk_ng, &c->d_blk_pair_off, &c->d_key, &c->d_key2, &c->d_val, &c->d_val2,
                    &c->d_rs_vrow, &c->d_rs_vtile, &c->d_rs_vtab, &c->d_rs_tab,
                    &c->d_sort_tmp, &c->d_node_row_off, &c->d_scalars, &c->d_nodes, &c->d_row_state, &c->d_row_cand,
                    &c->d_slab, &c->d_cand, &c->d_edges, &c->d_edges2, &c->d_edge_keys, &c->d_edge_keys2, &c->d_edge_w,
                    &c->d_edge_cnt, &c->d_nvalid, &c->d_edge_off, &c->d_edge_ng, &c->d_ba_in, &c->d_ba_blocks, &c->d_ba_out, &c->d_raw_blocks, &c->d_bkey, &c->d_bkey2, &c->d_bval, &c->d_bval2, &c->d_blk_rows, &c->d_vp_label, &c->d_vp_voff, &c->d_vp_vps, &c->d_vp_pts, &c->d_vp_off, &c->d_vp_labels, &c->d_vp_nc, &c->d_vp_ps, &c->d_vp_mat, &c->d_mg_in, &c->d_mg_out, &c->d_mg_edges, &c->d_gather, &c->d_vp_idx, &c->d_sfm_in, &c->d_sfm_keys, &c->d_sfm_keys2, &c->d_sfm_a, &c->d_sfm_b, &c->d_sfm_c, &c->d_sfm_d, &c->d_g_flag, &c->d_g_pos, &c->d_g_kc, &c->d_g_wc, &c->d_g_occ, &c->d_g_occ2, &c->d_g_hk, &c->d_g_hk2, &c->d_g_gidx, &c->d_g_gnode, &c->d_g_k1, &c->d_g_k1b, &c->d_g_k2, &c->d_g_k2b};
  for (DevBuf *b : bufs) b->release();
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->evk0) cudaEventDestroy(c->evk0);
  if (c->evk1) cudaEventDestroy(c->evk1);
  if (c->ev_raw) cudaEventDestroy(c->ev_raw);
  if (c->ev_scene) cudaEventDestroy(c->ev_scene);
  for (auto e : c->evk) cudaEventDestroy(e);
  for (auto &ch : c->chunks) cudaEventDestroy(ch.ev);
  for (auto e : c->event_pool) cudaEventDestroy(e);
  if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
  if (c->prep_stream) { cudaStreamSynchronize(c->prep_stream); cudaStreamDestroy(c->prep_stream); }
  if (c->out_stream) { cudaStreamSynchronize(c->out_stream); cudaStreamDestroy(c->out_stream); }
  for (auto e : c->evp) cudaEventDestroy(e);
  if (c->ev_run_begin) cudaEventDestroy(c->ev_run_begin);
  if (c->h_pin) cudaFreeHost(c->h_pin);
  if (c->h_ba_pin) cudaFreeHost(c->h_ba_pin);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

int lm_ctx_set_stream(lm_ctx *c, void *s) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = (cudaStream_t)s;
  c->own_stream = false;
  return LM_OK;
}
int lm_ctx_synchronize(lm_ctx *c) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->copy_stream));
  return sync_stream(c);
}

// Per-view constants (tri_kernels.cuh ViewT) from the reference's camera arrays.
static void make_view(int model_id, const double *kv, const double *qv, const double *t, lm::ViewD &d) {
  const double fx = kv[0], fy = kv[1], cx = kv[2], cy = kv[3];
  // CameraPose(qvec, tvec) normalises qvec (base/camera.h:92-93)
  M3h R = quat_to_R(qv);
  // K^-1 (closed form of Eigen's cofactor inverse for the pinhole K)
  const double ki[9] = {1.0 / fx, 0, -cx / fx, 0, 1.0 / fy, -cy / fy, 0, 0, 1};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) // M = R^T * Kinv
      d.M[3 * i + j] = R.m[0 * 3 + i] * ki[0 * 3 + j] + R.m[1 * 3 + i] * ki[1 * 3 + j] + R.m[2 * 3 + i] * ki[2 * 3 + j];
  for (int i = 0; i < 3; ++i) d.C[i] = -(R.m[0 * 3 + i] * t[0] + R.m[1 * 3 + i] * t[1] + R.m[2 * 3 + i] * t[2]);
  const double K[9] = {fx, 0, cx, 0, fy, cy, 0, 0, 1};
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j)
      d.P[4 * i + j] = K[3 * i] * R.m[j] + K[3 * i + 1] * R.m[3 + j] + K[3 * i + 2] * R.m[6 + j];
    d.P[4 * i + 3] = K[3 * i] * t[0] + K[3 * i + 1] * t[1] + K[3 * i + 2] * t[2];
  }
  d.fbar = (model_id == 0) ? fx : (fx + fy) / 2.0;
  d.pad = 0;
}

static int tri_clear_impl(lm_ctx *c, bool sync_copies);
static int upload_segs(lm_ctx *c, bool with_node_view) {
  // add_halfpix (base_line_triangulator.cc:32-43) is applied when both scene and config are known: on the device, from
  // the raw copy of the caller's segments, in stream order behind that copy.
  if (c->n_nodes)
    lm::launch_scene_prepare(c->d_segs_raw.as<double>(), c->n_nodes, (c->have_cfg && c->cfg.add_halfpix) ? 0.5 : 0.0,
                             c->d_line_off.as<int64_t>(), c->V, c->d_segs.as<double>(),
                             with_node_view ? c->d_node_view.as<uint16_t>() : nullptr, c->copy_stream);
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->ev_scene, c->copy_stream));
  return LM_OK;
}

int lm_scene_upload(lm_ctx *c, int32_t n_views, const int32_t *img_ids, const int32_t *model_ids, const double *kvec,
                    const double *qvec, const double *tvec, const int64_t *line_off, const double *segs) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (n_views <= 0 || n_views > 65535) return fail(LM_ERR_INVALID, "n_views must be in [1, 65535]");
  CU(cudaSetDevice(c->device));
  for (int v = 1; v < n_views; ++v)
    if (img_ids[v] <= img_ids[v - 1]) return fail(LM_ERR_INVALID, "img_ids must be strictly ascending");
  CU(cudaStreamSynchronize(c->copy_stream)); // the host staging tables below may still feed a previous upload
  CU(cudaStreamSynchronize(c->stream));      // ... and a previous run may still read buffers that get re-allocated
  c->V = n_views;
  c->img_ids.assign(img_ids, img_ids + n_views);
  c->id2view.clear();
  for (int v = 0; v < n_views; ++v) c->id2view[img_ids[v]] = v;
  c->line_off.assign(line_off, line_off + n_views + 1);
  c->n_nodes = line_off[n_views];
  if (c->n_nodes >= ((int64_t)1 << 31) - 64) return fail(LM_ERR_INVALID, "more than 2^31 2D lines in one scene");
  std::vector<lm::ViewD> &views = c->h_views;
  views.resize(n_views);
  for (int v = 0; v < n_views; ++v) {
    if (model_ids[v] != 0 && model_ids[v] != 1)
      return fail(LM_ERR_INVALID, "only SIMPLE_PINHOLE / PINHOLE are legal on this path (IsUndistorted check)");
    if (line_off[v + 1] - line_off[v] > 65535) return fail(LM_ERR_INVALID, "more than 65535 lines in one image");
    make_view(model_ids[v], kvec + 4 * v, qvec + 4 * v, tvec + 3 * v, views[v]);
  }
  CU(c->d_views.ensure(sizeof(lm::ViewD) * n_views));
  CU(c->d_node_view.ensure(std::max<size_t>(2, 2 * c->n_nodes)));
  CU(c->d_line_off.ensure(8 * (n_views + 1)));
  CU(c->d_segs_raw.ensure(std::max<size_t>(32, 32 * (size_t)c->n_nodes)));
  CU(c->d_segs.ensure(std::max<size_t>(32, 32 * (size_t)c->n_nodes)));
  CU(cudaMemcpyAsync(c->d_views.p, views.data(), sizeof(lm::ViewD) * n_views, cudaMemcpyHostToDevice, c->copy_stream));
  CU(cudaMemcpyAsync(c->d_line_off.p, c->line_off.data(), 8 * (n_views + 1), cudaMemcpyHostToDevice, c->copy_stream));
  CU(c->d_img_ids.ensure(4 * n_views));
  CU(cudaMemcpyAsync(c->d_img_ids.p, c->img_ids.data(), 4 * n_views, cudaMemcpyHostToDevice, c->copy_stream));
  // the 2D segments go up straight from the caller's buffer (a pinned buffer is not staged: it must stay unchanged until
  // the next call that synchronises, e.g. lm_tri_run; pageable memory is staged by the driver before this returns)
  if (c->n_nodes)
    CU(cudaMemcpyAsync(c->d_segs_raw.p, segs, 32 * (size_t)c->n_nodes, cudaMemcpyHostToDevice, c->copy_stream));
  c->have_scene = true;
  c->outside_shard_clean = false;
  int rc = upload_segs(c, true);
  if (rc) return rc;
  c->image_added.assign(n_views, 0);
  c->image_norder.assign(n_views, 0);
  c->stats.n_nodes = c->n_nodes;
  return tri_clear_impl(c, false); // (both streams were drained on entry: no match chunk is in flight)
}

int lm_tri_configure(lm_ctx *c, const lm_tri_config *cfg) {
  if (!c || !cfg) return fail(LM_ERR_INVALID, "NULL argument");
  if (cfg->merging_strategy != 0)
    return fail(LM_ERR_INVALID, "Error!The given merging strategy is not implemented"); // global_line_triangulator.cc:318
  const bool halfpix_changed = !c->have_cfg || (c->cfg.add_halfpix != cfg->add_halfpix);
  c->cfg = *cfg;
  c->have_cfg = true;
  c->ran = false;
  if (c->have_scene && halfpix_changed) return upload_segs(c, false);
  return LM_OK;
}
int lm_tri_set_ranges(lm_ctx *c, const double lo[3], const double hi[3]) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  c->ranges_flag = true;
  for (int i = 0; i < 3; ++i) { c->rlo[i] = lo[i]; c->rhi[i] = hi[i]; }
  c->ran = false;
  return LM_OK;
}
int lm_tri_unset_ranges(lm_ctx *c) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  c->ranges_flag = false;
  c->ran = false;
  return LM_OK;
}
int lm_tri_set_vps(lm_ctx *c, int32_t n_images, const int32_t *img_ids, const int64_t *label_off, const int32_t *labels,
                   const int64_t *vp_off, const double *vps) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (!c->have_scene) return fail(LM_ERR_STATE, "lm_scene_upload must precede InitVPResults");
  CU(cudaSetDevice(c->device));
  std::vector<int32_t> lab(std::max<int64_t>(c->n_nodes, 1), -1);
  std::vector<int64_t> voff(c->V + 1, 0);
  std::vector<int64_t> cnt(c->V, 0);
  std::vector<int> src(c->V, -1);
  for (int i = 0; i < n_images; ++i) {
    auto it = c->id2view.find(img_ids[i]);
    if (it == c->id2view.end()) return fail(LM_ERR_INVALID, "unknown image id in InitVPResults");
    const int v = it->second;
    const int64_t nl = label_off[i + 1] - label_off[i];
    if (nl != c->line_off[v + 1] - c->line_off[v]) return fail(LM_ERR_INVALID, "VPResult.labels size != number of lines");
    cnt[v] = vp_off[i + 1] - vp_off[i];
    src[v] = i;
    for (int64_t l = 0; l < nl; ++l) {
      const int32_t x = labels[label_off[i] + l];
      if (x >= cnt[v]) return fail(LM_ERR_INVALID, "VP label out of range");
      lab[c->line_off[v] + l] = x;
    }
  }
  for (int v = 0; v < c->V; ++v) voff[v + 1] = voff[v] + cnt[v];
  std::vector<double> vv(3 * std::max<int64_t>(voff[c->V], 1), 0.0);
  for (int v = 0; v < c->V; ++v)
    if (src[v] >= 0)
      memcpy(&vv[3 * voff[v]], vps + 3 * vp_off[src[v]], 24 * cnt[v]);
  CU(cudaStreamSynchronize(c->stream)); // a previous run may still read the tables that are re-allocated
  CU(c->d_vp_label.ensure(4 * lab.size()));
  CU(c->d_vp_voff.ensure(8 * voff.size()));
  CU(c->d_vp_vps.ensure(8 * vv.size()));
  CU(cudaMemcpyAsync(c->d_vp_label.p, lab.data(), 4 * lab.size(), cudaMemcpyHostToDevice, c->copy_stream));
  CU(cudaMemcpyAsync(c->d_vp_voff.p, voff.data(), 8 * voff.size(), cudaMemcpyHostToDevice, c->copy_stream));
  CU(cudaMemcpyAsync(c->d_vp_vps.p, vv.data(), 8 * vv.size(), cudaMemcpyHostToDevice, c->copy_stream));
  CU(cudaEventRecord(c->ev_scene, c->copy_stream));
  CU(cudaStreamSynchronize(c->copy_stream)); // the staging vectors die here
  c->have_vps = true;
  c->ran = false;
  return LM_OK;
}

int lm_tri_clear(lm_ctx *c) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  return tri_clear_impl(c, true);
}
static int tri_clear_impl(lm_ctx *c, bool sync_copies) {
  c->blocks.clear();
  c->raw_uploaded = 0;
  std::fill(c->image_added.begin(), c->image_added.end(), 0);
  std::fill(c->image_norder.begin(), c->image_norder.end(), 0);
  if (c->copy_stream && sync_copies) cudaStreamSynchronize(c->copy_stream); // (the chunk events go back to the pool)
  for (auto &ch : c->chunks) c->event_pool.push_back(ch.ev);
  c->chunks.clear();
  c->pairs_rows = 0;
  c->any_exhaustive = c->any_matches = false;
  c->ran = false;
  c->h_nodes_valid = c->h_rows_valid = c->h_edges_valid = false;
  c->edges_collected = false;
  c->tracks.clear();
  c->graph_nodes.clear();
  return LM_OK;
}
int lm_tri_set_node_sink(lm_ctx *c, void *host_nodes) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  c->node_sink = static_cast<char *>(host_nodes);
  return LM_OK;
}
int lm_tri_set_pipeline_groups(lm_ctx *c, int32_t n) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (n < 1 || n > 64) return fail(LM_ERR_INVALID, "pipeline groups must be in [1, 64]");
  c->pipeline_groups = n;
  return LM_OK;
}

int lm_tri_set_shard(lm_ctx *c, int32_t b, int32_t e) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (b != c->shard_begin || e != c->shard_end) c->outside_shard_clean = false;
  c->shard_begin = b;
  c->shard_end = e;
  c->ran = false;
  return LM_OK;
}

// Mirror the block descriptors added since the last call on the device (copy stream, ahead of their matches).
static int upload_raw_blocks(lm_ctx *c) {
  const int64_t n = (int64_t)c->blocks.size();
  if (n <= c->raw_uploaded) return LM_OK;
  if ((size_t)n * sizeof(lm::RawBlock) > c->d_raw_blocks.cap) {
    CU(cudaStreamSynchronize(c->copy_stream));
    CU(cudaStreamSynchronize(c->stream));
    DevBuf nbuf;
    CU(nbuf.ensure(std::max<size_t>((size_t)n * sizeof(lm::RawBlock) * 2, 1 << 16)));
    if (c->raw_uploaded)
      CU(cudaMemcpy(nbuf.p, c->d_raw_blocks.p, c->raw_uploaded * sizeof(lm::RawBlock), cudaMemcpyDeviceToDevice));
    c->d_raw_blocks.release();
    c->d_raw_blocks = nbuf;
  }
  std::vector<lm::RawBlock> tmp(n - c->raw_uploaded);
  for (int64_t i = c->raw_uploaded; i < n; ++i) {
    const MatchBlock &b = c->blocks[i];
    lm::RawBlock &r = tmp[i - c->raw_uploaded];
    r.src_view = b.src_view; r.ng_view = b.ng_view; r.n_rows = b.n_rows; r.pair_off = b.pair_off; r.order = b.order; r.pad = 0;
  }
  // pageable source: the runtime stages it, so `tmp` may die at scope exit
  CU(cudaMemcpyAsync(c->d_raw_blocks.as<lm::RawBlock>() + c->raw_uploaded, tmp.data(), tmp.size() * sizeof(lm::RawBlock),
                     cudaMemcpyHostToDevice, c->copy_stream));
  if (!c->ev_raw) CU(cudaEventCreateWithFlags(&c->ev_raw, cudaEventDisableTiming));
  CU(cudaEventRecord(c->ev_raw, c->copy_stream));
  c->raw_uploaded = n;
  return LM_OK;
}

// Upload `total` match rows into the device store in chunks, one event per chunk, on the copy stream.
static int upload_pairs(lm_ctx *c, const int32_t *pairs, int64_t total, bool on_device) {
  if ((size_t)(c->pairs_rows + total) * 8 > c->d_pairs.cap) {
    CU(cudaStreamSynchronize(c->copy_stream));
    DevBuf nbuf;
    CU(nbuf.ensure(std::max<size_t>((size_t)(c->pairs_rows + total) * 8 * 2, 1 << 20)));
    if (c->pairs_rows) CU(cudaMemcpyAsync(nbuf.p, c->d_pairs.p, c->pairs_rows * 8, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->d_pairs.release();
    c->d_pairs = nbuf;
  }
  // one event per copy; the copies start at 2 MB and double up to 16 MB, so that the first pipeline group of a run (a few
  // per cent of the rows) does not wait for a full-size chunk
  const int64_t kChunk = 2 << 20, kEventEvery = 1;
  int64_t k = 0, step = 256 << 10;
  for (int64_t o = 0, n = 0; o < total; o += n, ++k, step = std::min(kChunk, step * 2)) {
    n = std::min(step, total - o);
    CU(cudaMemcpyAsync(c->d_pairs.as<char>() + (c->pairs_rows + o) * 8, pairs + 2 * o, n * 8,
                       on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->copy_stream));
    if ((k + 1) % kEventEvery == 0 || o + n >= total) {
      cudaEvent_t ev;
      if (!c->event_pool.empty()) { ev = c->event_pool.back(); c->event_pool.pop_back(); }
      else CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      CU(cudaEventRecord(ev, c->copy_stream));
      c->chunks.push_back({c->pairs_rows + o + n, ev});
    }
  }
  return LM_OK;
}

static int add_matches_impl(lm_ctx *c, int32_t img_id, int32_t n_ng, const int32_t *ng_ids, const int64_t *row_off,
                            const int32_t *pairs, bool on_device) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (!c->have_scene) return fail(LM_ERR_STATE, "lm_scene_upload must precede TriangulateImage");
  CU(cudaSetDevice(c->device));
  auto it = c->id2view.find(img_id);
  if (it == c->id2view.end()) return fail(LM_ERR_INVALID, "unknown image id " + std::to_string(img_id));
  const int sv = it->second;
  if (c->image_added[sv]) return fail(LM_ERR_STATE, "image " + std::to_string(img_id) + " was already triangulated");
  if (c->any_exhaustive) return fail(LM_ERR_STATE, "cannot mix exhaustive and match-based triangulation in one run");
  const int64_t total = n_ng > 0 ? row_off[n_ng] : 0;
  std::set<int> seen;
  for (int g = 0; g < n_ng; ++g) {
    if (c->id2view.find(ng_ids[g]) == c->id2view.end())
      return fail(LM_ERR_INVALID, "unknown neighbor image id " + std::to_string(ng_ids[g]));
    if (!seen.insert(ng_ids[g]).second) return fail(LM_ERR_INVALID, "duplicate neighbor id in one TriangulateImage call");
    if (row_off[g + 1] < row_off[g]) return fail(LM_ERR_INVALID, "row_off must be non-decreasing");
  }
  for (int g = 0; g < n_ng; ++g) {
    MatchBlock b;
    b.src_view = sv;
    b.ng_view = c->id2view[ng_ids[g]];
    b.n_rows = row_off[g + 1] - row_off[g];
    b.pair_off = c->pairs_rows + row_off[g];
    b.order = 0; // std::map order = ascending neighbour id (base_line_triangulator.cc:74)
    c->blocks.push_back(b);
  }
  {
    int rc_ = upload_raw_blocks(c);
    if (!rc_) rc_ = upload_pairs(c, pairs, total, on_device);
    if (rc_) return rc_;
  }
  c->pairs_rows += total;
  c->image_added[sv] = 1;
  c->any_matches = true;
  c->ran = false;
  return LM_OK;
}
int lm_tri_add_image_matches(lm_ctx *c, int32_t img_id, int32_t n_ng, const int32_t *ng_ids, const int64_t *row_off,
                             const int32_t *pairs) {
  return add_matches_impl(c, img_id, n_ng, ng_ids, row_off, pairs, false);
}
int lm_tri_add_image_matches_device(lm_ctx *c, int32_t img_id, int32_t n_ng, const int32_t *ng_ids,
                                    const int64_t *row_off, const int32_t *d_pairs) {
  return add_matches_impl(c, img_id, n_ng, ng_ids, row_off, d_pairs, true);
}
int lm_tri_add_matches_bulk(lm_ctx *c, int32_t n_blocks, const int32_t *src_img_ids, const int32_t *ng_img_ids,
                            const int64_t *row_off, const int32_t *pairs) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (!c->have_scene) return fail(LM_ERR_STATE, "lm_scene_upload must precede TriangulateImage");
  if (c->any_exhaustive) return fail(LM_ERR_STATE, "cannot mix exhaustive and match-based triangulation in one run");
  CU(cudaSetDevice(c->device));
  const int64_t total = n_blocks > 0 ? row_off[n_blocks] : 0;
  std::vector<char> seen_img(c->V, 0);
  std::vector<MatchBlock> nb;
  nb.reserve(n_blocks);
  for (int b = 0; b < n_blocks; ++b) {
    auto is = c->id2view.find(src_img_ids[b]), in_ = c->id2view.find(ng_img_ids[b]);
    if (is == c->id2view.end() || in_ == c->id2view.end()) return fail(LM_ERR_INVALID, "unknown image id in matches");
    if (c->image_added[is->second]) return fail(LM_ERR_STATE, "image " + std::to_string(src_img_ids[b]) + " was already triangulated");
    if (row_off[b + 1] < row_off[b]) return fail(LM_ERR_INVALID, "row_off must be non-decreasing");
    seen_img[is->second] = 1;
    MatchBlock m;
    m.src_view = is->second; m.ng_view = in_->second; m.n_rows = row_off[b + 1] - row_off[b];
    m.pair_off = c->pairs_rows + row_off[b]; m.order = 0;
    nb.push_back(m);
  }
  c->blocks.insert(c->blocks.end(), nb.begin(), nb.end());
  {
    int rc_ = upload_raw_blocks(c);
    if (!rc_) rc_ = upload_pairs(c, pairs, total, false);
    if (rc_) return rc_;
  }
  c->pairs_rows += total;
  for (int v = 0; v < c->V; ++v) if (seen_img[v]) c->image_added[v] = 1;
  c->any_matches = true;
  c->ran = false;
  return LM_OK;
}

int lm_tri_get_nodes(lm_ctx *c, lm_node_record *out) {
  if (!c || !out) return fail(LM_ERR_INVALID, "NULL argument");
  int rc = ensure_ran(c);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out, c->d_nodes.p, sizeof(lm::NodeRecord) * c->n_nodes, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return LM_OK;
}

int64_t lm_tri_get_all_valid_edges(lm_ctx *c, int64_t *node_off, int32_t *edges) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  int rc = ensure_ran(c);
  if (rc) return rc;
  const int64_t ne = c->stats.n_valid_edges;
  if (!node_off && !edges) return ne;
  // converted on the device and copied straight into the caller's buffers (pinned buffers avoid staging)
  const int64_t nsh = c->node_end - c->node_begin;
  if (nsh <= 0) { // empty shard: nothing on the device to convert
    if (node_off) memset(node_off, 0, 8 * (size_t)(c->n_nodes + 1));
    return 0;
  }
  const size_t off_bytes = 8 * (size_t)(c->n_nodes + 1), pair_bytes = 8 * (size_t)std::max<int64_t>(ne, 1);
  CU(c->d_host_edges.ensure(off_bytes + pair_bytes + 256));
  int64_t *d_off = c->d_host_edges.as<int64_t>();
  int32_t *d_pairs = reinterpret_cast<int32_t *>(c->d_host_edges.as<char>() + ((off_bytes + 255) / 256) * 256);
  lm::launch_edges_for_host(c->d_edge_off.as<uint32_t>(), c->d_edge_ng.as<uint32_t>(), c->d_img_ids.as<int32_t>(), nsh,
                            ne, c->node_begin, c->n_nodes, d_off, d_pairs, c->stream);
  c->stats.n_kernel_launches += 1;
  if (node_off) CU(cudaMemcpyAsync(node_off, d_off, off_bytes, cudaMemcpyDeviceToHost, c->stream));
  if (edges && ne) CU(cudaMemcpyAsync(edges, d_pairs, 8 * (size_t)ne, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return ne;
}

int lm_tri_add_image_exhaustive(lm_ctx *c, int32_t img_id, int32_t n_ng, const int32_t *ng_ids) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (!c->have_scene) return fail(LM_ERR_STATE, "lm_scene_upload must precede TriangulateImageExhaustiveMatch");
  auto it = c->id2view.find(img_id);
  if (it == c->id2view.end()) return fail(LM_ERR_INVALID, "unknown image id " + std::to_string(img_id));
  const int sv = it->second;
  if (c->image_added[sv]) return fail(LM_ERR_STATE, "image " + std::to_string(img_id) + " was already triangulated");
  if (c->any_matches) return fail(LM_ERR_STATE, "cannot mix exhaustive and match-based triangulation in one run");
  const int64_t nl = c->line_off[sv + 1] - c->line_off[sv];
  for (int g = 0; g < n_ng; ++g) {
    auto f = c->id2view.find(ng_ids[g]);
    if (f == c->id2view.end()) return fail(LM_ERR_INVALID, "unknown neighbor image id " + std::to_string(ng_ids[g]));
    MatchBlock b;
    b.src_view = sv;
    b.ng_view = f->second;
    b.n_rows = nl * (c->line_off[b.ng_view + 1] - c->line_off[b.ng_view]);
    b.pair_off = -1;
    b.order = g; // neighbours are visited in the given order (base_line_triangulator.cc:116-117)
    c->blocks.push_back(b);
  }
  c->image_added[sv] = 1;
  c->any_exhaustive = true;
  c->ran = false;
  return upload_raw_blocks(c);
}

int lm_tri_run(lm_ctx *c) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (!c->have_scene) return fail(LM_ERR_STATE, "no scene uploaded");
  if (!c->have_cfg) return fail(LM_ERR_STATE, "lm_tri_configure must precede lm_tri_run");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const int vb = std::max(0, c->shard_begin), ve = (c->shard_end < 0) ? c->V : std::min(c->V, c->shard_end);
  // blocks of this shard in flat order: (source view, neighbour order)
  std::vector<MatchBlock> blk;
  for (const MatchBlock &b : c->blocks)
    if (b.src_view >= vb && b.src_view < ve) blk.push_back(b);
  const bool exhaustive = c->any_exhaustive;
  std::stable_sort(blk.begin(), blk.end(), [exhaustive](const MatchBlock &a, const MatchBlock &b) {
    if (a.src_view != b.src_view) return a.src_view < b.src_view;
    if (exhaustive) return a.order < b.order;
    return a.ng_view < b.ng_view;
  });
  const int nb = (int)blk.size();
  std::vector<int64_t> row_off(nb + 1, 0), pair_off(nb);
  std::vector<int32_t> bsrc(nb), bng(nb);
  for (int i = 0; i < nb; ++i) {
    row_off[i + 1] = row_off[i] + blk[i].n_rows;
    pair_off[i] = blk[i].pair_off;
    bsrc[i] = blk[i].src_view;
    bng[i] = blk[i].ng_view;
  }
  const int64_t n_rows = row_off[nb];
  // the sort and scan item counts are 32-bit signed
  if (n_rows >= ((int64_t)1 << 31) - 64) return fail(LM_ERR_INVALID, "more than 2^31 match rows in one run (shard the scene by source image)");
  c->n_rows = n_rows;
  c->node_begin = c->line_off[vb];
  c->node_end = c->line_off[ve];
  c->h_nodes_valid = c->h_rows_valid = c->h_edges_valid = false;
  c->edges_collected = false;
  c->edges_count_on_device = false;
  c->tracks.clear();

  CU(c->d_blk_row_off.ensure(8 * (nb + 1)));
  CU(c->d_blk_src.ensure(4 * std::max(nb + 1, 2)));
  CU(c->d_blk_ng.ensure(4 * std::max(nb + 1, 2)));
  CU(c->d_blk_pair_off.ensure(8 * std::max(nb, 1)));
  CU(c->d_key2.ensure(4 * std::max<int64_t>(n_rows, 1)));
  CU(c->d_val2.ensure(4 * std::max<int64_t>(n_rows, 1)));
  CU(c->d_node_row_off.ensure(4 * (c->n_nodes + 2)));
  CU(c->d_scalars.ensure(1024));
  CU(c->d_nodes.ensure(sizeof(lm::NodeRecord) * std::max<int64_t>(c->n_nodes, 1)));
  const int ns = (c->cfg.use_vp && !c->cfg.disable_vp_triangulation && c->have_vps) ? 3 : 1;
  c->ns = ns;
  CU(c->d_row_state.ensure(std::max<int64_t>(n_rows * ns, 1)));
  if (c->cfg.debug_mode) CU(c->d_row_cand.ensure(80 * std::max<int64_t>(n_rows * ns, 1)));

#ifdef LM_TRACE
  const auto lm_t0 = std::chrono::steady_clock::now();
  auto lm_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - lm_t0).count(); };
#endif
  CU(cudaEventRecord(c->ev0, s));
#ifdef LM_TRACE
  cudaEventSynchronize(c->ev0);
  fprintf(stderr, "[lm trace] ev0 executed %.3f ms after run entry\n", lm_ms());
#endif
  // Two compute streams: `sp` prepares the rows of a pipeline group (expansion, sort, node offsets), `s` runs the node
  // kernels. The preparation of group g+1 is queued right behind that of group g, so it executes under the node kernel of
  // group g; everything `sp` touches is per-group slices, its own scratch, or is read by `s` only after the group's event.
  cudaStream_t sp = c->prep_stream;
  CU(cudaEventRecord(c->ev_run_begin, s)); // whatever the caller queued on the engine's stream comes first
  CU(cudaStreamWaitEvent(sp, c->ev_run_begin, 0));
  // scene tables / VP tables travel on the copy stream (see lm_ctx::ev_scene)
  CU(cudaStreamWaitEvent(sp, c->ev_scene, 0));
  CU(cudaStreamWaitEvent(s, c->ev_scene, 0));
  lm::launch_zero_words(c->d_scalars.p, 256, sp);
  // block tables, derived on the device from the descriptors uploaded with the matches (no transfer now)
  {
    const int n_all = (int)c->blocks.size();
    CU(c->d_blk_rows.ensure(8 * (nb + 2)));
    if (n_all) {
      CU(c->d_bkey.ensure(4 * n_all)); CU(c->d_bkey2.ensure(4 * n_all));
      CU(c->d_bval.ensure(4 * n_all)); CU(c->d_bval2.ensure(4 * n_all));
      // the descriptors travel on the copy stream ahead of their matches (bulk add: ahead of all matches)
      if (c->ev_raw) CU(cudaStreamWaitEvent(sp, c->ev_raw, 0));
      lm::launch_block_keys(c->d_raw_blocks.as<lm::RawBlock>(), n_all, vb, ve, exhaustive ? 1 : 0, c->d_bkey.as<uint32_t>(),
                            c->d_bval.as<uint32_t>(), sp);
      cub::DoubleBuffer<uint32_t> bk(c->d_bkey.as<uint32_t>(), c->d_bkey2.as<uint32_t>());
      cub::DoubleBuffer<uint32_t> bv(c->d_bval.as<uint32_t>(), c->d_bval2.as<uint32_t>());
      size_t tmpb = 0;
      CU(cub::DeviceRadixSort::SortPairs(nullptr, tmpb, bk, bv, n_all, 0, 32, sp));
      CU(c->d_sort_tmp.ensure(tmpb));
      CU(cub::DeviceRadixSort::SortPairs(c->d_sort_tmp.p, tmpb, bk, bv, n_all, 0, 32, sp));
      lm::launch_block_gather(c->d_raw_blocks.as<lm::RawBlock>(), bv.Current(), nb, c->d_blk_src.as<int32_t>(),
                              c->d_blk_ng.as<int32_t>(), c->d_blk_pair_off.as<int64_t>(), c->d_blk_rows.as<int64_t>(), sp);
    } else {
      lm::launch_zero_words(c->d_blk_rows.p, 4, sp);
    }
    size_t tmps = 0;
    CU(cub::DeviceScan::ExclusiveSum(nullptr, tmps, c->d_blk_rows.as<int64_t>(), c->d_blk_row_off.as<int64_t>(), nb + 1, sp));
    CU(c->d_sort_tmp.ensure(tmps));
    CU(cub::DeviceScan::ExclusiveSum(c->d_sort_tmp.p, tmps, c->d_blk_rows.as<int64_t>(), c->d_blk_row_off.as<int64_t>(),
                                     nb + 1, sp));
  }
  // d_scalars words: [1] index error, [2] staging overflow, [3] largest candidate count of a node (split path), bytes
  // 16..47 counters, words [16 + g] largest node of group g
  int *d_err = c->d_scalars.as<int>() + 1;
  unsigned long long *d_counters = reinterpret_cast<unsigned long long *>(c->d_scalars.as<char>() + 16);
  int launches = 0;
  lm::TriParams p;
  memset(&p, 0, sizeof(p));
  p.views = c->d_views.as<lm::ViewD>();
  p.segs = c->d_segs.as<double4>();
  p.node_view = c->d_node_view.as<uint16_t>();
  p.line_off = c->d_line_off.as<int64_t>();
  p.node_row_off = c->d_node_row_off.as<uint32_t>();
  p.nodes = c->d_nodes.as<lm::NodeRecord>();
  p.row_state = c->d_row_state.as<uint8_t>();
  p.row_cand = c->cfg.debug_mode ? c->d_row_cand.as<double>() : nullptr;
  p.counters = d_counters;
  p.overflow = c->d_scalars.as<int>() + 2;
  p.max_cand = c->d_scalars.as<unsigned int>() + 3;
  p.node_begin = c->node_begin;
  p.node_end = c->node_end;
  const lm_tri_config &g = c->cfg;
  p.min_length_2d = g.min_length_2d; p.line_tri_angle_threshold = g.line_tri_angle_threshold;
  p.IoU_threshold = g.IoU_threshold; p.sensitivity_threshold = g.sensitivity_threshold; p.var2d = g.var2d;
  p.fullscore_th = g.fullscore_th; p.max_valid_conns = g.max_valid_conns;
  p.use_endpoints_triangulation = g.use_endpoints_triangulation; p.disable_algebraic = g.disable_algebraic_triangulation;
  p.use_vp = (ns == 3); p.disable_vp = g.disable_vp_triangulation;
  p.vp_label = c->d_vp_label.as<int32_t>(); p.vp_off = c->d_vp_voff.as<int64_t>(); p.vps = c->d_vp_vps.as<double>();
  p.ranges_flag = c->ranges_flag;
  for (int i = 0; i < 3; ++i) { p.rlo[i] = c->rlo[i]; p.rhi[i] = c->rhi[i]; }
  p.l2d = to_dev<double>(g.linker2d);
  {
    lm_linker_config l3 = g.linker3d; // set_to_shared_parent_scoring (line_linker.h:115-121)
    l3.use_angle = 1; l3.use_overlap = 0; l3.use_perp = 0; l3.use_innerseg = 0; l3.use_scaleinv = 1;
    p.l3d = to_dev<double>(l3);
  }
  {
    const double kPi = 3.14159265358979323846;
    const double t3 = p.l3d.th_angle, t2 = p.l2d.th_angle;
    p.cos_th3d_f = (t3 >= 90.0) ? -1.0f : (float)(std::cos(t3 * kPi / 180.0) - 4e-6);
    const double c2 = (t2 >= 90.0) ? 0.0 : std::cos(t2 * kPi / 180.0);
    p.cos2_th2d = c2 * c2;
    p.th_perp2_2d = p.l2d.th_perp * p.l2d.th_perp;
    const double ta = p.line_tri_angle_threshold, tsn = p.sensitivity_threshold;
    p.tri_poly_ok = (ta > 0.0 && ta < 90.0);
    p.sens_poly_ok = (tsn > 0.0 && tsn < 90.0);
    p.sin2_tri = std::sin(ta * kPi / 180.0) * std::sin(ta * kPi / 180.0);
    p.sin2_sens = std::sin(tsn * kPi / 180.0) * std::sin(tsn * kPi / 180.0);
    p.fast_forms = (p.l2d.use_innerseg || getenv("LIMAP_B200_REFERENCE_FORMS")) ? 0 : 1;
    p.inv_sig_a3 = 1.0 / (p.l3d.th_angle * p.l3d.mult);
    p.inv_sig_s3 = 1.0 / (p.l3d.th_scaleinv * p.l3d.mult);
    p.inv_sig_a2 = 1.0 / (p.l2d.th_angle * p.l2d.mult);
    p.inv_sig_p2 = 1.0 / (p.l2d.th_perp * p.l2d.mult);
    p.q_cut3 = -2.0 * std::log(p.l3d.score_th) * (1.0 + 1e-9);
    p.q_cut3_lo = -2.0 * std::log(p.l3d.score_th) * (1.0 - 1e-9);
    p.q_cut2 = -2.0 * std::log(p.l2d.score_th) * (1.0 + 1e-9);
    p.q_cut2_lo = -2.0 * std::log(p.l2d.score_th) * (1.0 - 1e-9);
    p.inv_smart_den2 = 1.0 / (p.l2d.th_smartoverlap - p.l2d.th_overlap);
  }
  // ---- groups of source images: sort + node kernel of group g overlap the upload of group g+1 -----------
  int nbits = 1;
  while (((int64_t)1 << nbits) < c->n_nodes) ++nbits;
  // canonical sorted buffers: d_key2 / d_val2
  c->sorted_key = c->d_key2.as<uint32_t>();
  c->sorted_val = c->d_val2.as<uint32_t>();
  p.row_ng = c->sorted_val;
  const int n_groups = exhaustive ? 1 : (int)std::max<int64_t>(1, std::min<int64_t>(c->pipeline_groups, n_rows >> 16));
  c->node_kernel_ms_acc = 0;
  int bg0 = 0, gv0 = vb;
  const int64_t n_shard_nodes = c->node_end - c->node_begin;
  // Results outside the shard (filled by lm_tri_import_nodes in a multi-GPU run) start from the empty record, so a
  // getter never sees uninitialised memory; done once per scene/shard, imports survive later runs.
  if (!c->outside_shard_clean && (c->node_begin > 0 || c->node_end < c->n_nodes)) {
    if (c->node_begin > 0) {
      CU(cudaMemsetAsync(c->d_nodes.p, 0, sizeof(lm::NodeRecord) * c->node_begin, s));
      CU(cudaMemsetAsync(c->d_node_row_off.p, 0, 4 * c->node_begin, s));
    }
    if (c->node_end < c->n_nodes) {
      CU(cudaMemsetAsync(c->d_nodes.as<lm::NodeRecord>() + c->node_end, 0, sizeof(lm::NodeRecord) * (c->n_nodes - c->node_end), s));
      CU(cudaMemsetAsync(c->d_node_row_off.as<uint32_t>() + c->node_end + 1, 0, 4 * (c->n_nodes - c->node_end), s));
    }
    c->outside_shard_clean = true;
  }
  // The staging capacity of the node kernel (candidates per node held in shared memory) comes from the previous run
  // (default: what four CTAs per SM allow); the kernel flags nodes that do not fit and the run is repeated once with
  // the exact size. No read-back, no host synchronisation until everything of this run is queued.
  const bool fast_kernel = p.fast_forms && !p.use_endpoints_triangulation;
  const size_t smem_limit = (size_t)std::max(0, c->max_smem_optin - 1024);
  int cap = c->cap_hint > 0 ? c->cap_hint : 224;
  if (exhaustive && c->cap_hint == 0) { // every node sees all lines of every neighbour: known on the host
    int64_t mr = 0, cur = 0;
    int cur_src = -1;
    for (int i = 0; i < nb; ++i) {
      if (blk[i].src_view != cur_src) { cur_src = blk[i].src_view; cur = 0; }
      cur += c->line_off[blk[i].ng_view + 1] - c->line_off[blk[i].ng_view];
      mr = std::max(mr, cur);
    }
    if (mr * ns > 65535) return fail(LM_ERR_INVALID, "more than 65535 candidates possible for one 2D line");
    cap = 32;
    while (cap < mr * ns) cap += 32;
  }
  while ((int)c->evk.size() < 2 * n_groups) {
    cudaEvent_t e;
    CU(cudaEventCreate(&e));
    c->evk.push_back(e);
  }
  while ((int)c->evp.size() < n_groups) {
    cudaEvent_t e;
    CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    c->evp.push_back(e);
  }
  // Split form of the fast path (tri_gen_kernel + tri_score_kernel, the default): its staging capacity comes from the
  // largest candidate count of a node, which the score kernel reports; LIMAP_B200_TRI_FUSED=1 (read per run) selects the
  // fused tri_node_kernel. Exhaustive matching and the generic forms always run fused.
  const int cap_split = c->cap_hint_cand > 0 ? c->cap_hint_cand : cap;
  const bool split = fast_kernel && !exhaustive && !getenv("LIMAP_B200_TRI_FUSED") &&
                     lm::tri_score_smem_bytes(cap_split) <= smem_limit;
  // blocks [gb[g], gb[g + 1]) with whole source images form group g
  std::vector<int> gb(n_groups + 1, nb);
  gb[0] = 0;
  int64_t max_group_rows = 0;
  for (int g = 0; g < n_groups; ++g) {
    int bg1 = nb;
    if (g + 1 < n_groups) {
      // small groups at both ends (smoothstep): the first one is the only one whose matches nothing else can hide, the
      // last one is the only one whose results nothing else can hide
      const double tg = (g + 1.0) / n_groups;
      const int64_t target = (int64_t)((double)n_rows * (tg * tg * (3.0 - 2.0 * tg)));
      bg1 = gb[g];
      while (bg1 < nb && row_off[bg1] < target) ++bg1;
      while (bg1 < nb && bg1 > 0 && blk[bg1].src_view == blk[bg1 - 1].src_view) ++bg1; // finish the image
    }
    gb[g + 1] = bg1;
    max_group_rows = std::max(max_group_rows, row_off[bg1] - row_off[gb[g]]);
  }
  // Node-major rows: a per-view stable counting sort (row_count / row_scan / row_scatter) by default; views with more
  // than kRowSortMaxLines lines, exhaustive matching and LIMAP_B200_ROW_SORT=cub (read per run) take the radix-sort
  // path (expand_rows -> stable radix sort by node id -> node_offsets). Both give the same rows and node offsets.
  const char *row_sort_env = getenv("LIMAP_B200_ROW_SORT");
  const bool row_sort_cub = exhaustive || (row_sort_env && !strcmp(row_sort_env, "cub"));
  const int nvs = ve - vb;
  // host copy of what row_views_kernel derives on the device: first row and first tile of every view of the shard
  std::vector<int64_t> vrow(nvs + 1, 0);
  std::vector<int32_t> vtile(nvs + 1, 0);
  bool any_radix_rows = row_sort_cub && n_rows > 0;
  if (!row_sort_cub) {
    for (int i = 0; i < nb; ++i) vrow[blk[i].src_view - vb + 1] += blk[i].n_rows;
    int64_t tab_words = 0;
    for (int i = 0; i < nvs; ++i) {
      const int64_t L = c->line_off[vb + i + 1] - c->line_off[vb + i], rows = vrow[i + 1];
      const int64_t nt = L <= lm::kRowSortMaxLines ? (rows + lm::kRowSortTile - 1) / lm::kRowSortTile : 0;
      if (L > lm::kRowSortMaxLines && rows > 0) any_radix_rows = true;
      vtile[i + 1] = vtile[i] + (int32_t)nt;
      tab_words += nt * std::max<int64_t>(L, 1);
      vrow[i + 1] += vrow[i];
    }
    CU(c->d_rs_vrow.ensure(8 * (nvs + 1)));
    CU(c->d_rs_vtile.ensure(4 * (nvs + 1)));
    CU(c->d_rs_vtab.ensure(8 * (nvs + 1)));
    CU(c->d_rs_tab.ensure(4 * std::max<int64_t>(tab_words, 1)));
    lm::launch_row_views(c->d_blk_row_off.as<int64_t>(), c->d_blk_src.as<int32_t>(), nb, c->d_line_off.as<int64_t>(), vb,
                         nvs, c->d_rs_vrow.as<int64_t>(), c->d_rs_vtile.as<int32_t>(), c->d_rs_vtab.as<int64_t>(), sp);
    ++launches;
  }
  if (any_radix_rows) {
    CU(c->d_key.ensure(4 * std::max<int64_t>(n_rows, 1)));
    CU(c->d_val.ensure(4 * std::max<int64_t>(n_rows, 1)));
  }
  // stable LSD radix sort by node id of rows [r0, r1) into d_key2 / d_val2 keeps (neighbour, row) order inside every node
  auto radix_sort_rows = [&](int64_t r0, int64_t r1) -> cudaError_t {
    cub::DoubleBuffer<uint32_t> dk(c->d_key.as<uint32_t>() + r0, c->d_key2.as<uint32_t>() + r0);
    cub::DoubleBuffer<uint32_t> dv(c->d_val.as<uint32_t>() + r0, c->d_val2.as<uint32_t>() + r0);
    size_t tmp = 0;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, tmp, dk, dv, (int)(r1 - r0), 0, nbits, sp);
    if (e == cudaSuccess) e = c->d_sort_tmp.ensure(tmp);
    if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(c->d_sort_tmp.p, tmp, dk, dv, (int)(r1 - r0), 0, nbits, sp);
    launches += (nbits + 7) / 8 + 1;
    if (e == cudaSuccess && dk.Current() != c->d_key2.as<uint32_t>() + r0) {
      e = cudaMemcpyAsync(c->d_key2.as<uint32_t>() + r0, dk.Current(), 4 * (r1 - r0), cudaMemcpyDeviceToDevice, sp);
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(c->d_val2.as<uint32_t>() + r0, dv.Current(), 4 * (r1 - r0), cudaMemcpyDeviceToDevice, sp);
    }
    return e;
  };
  if (split) {
    p.row_node = c->sorted_key;
    p.cand_stride = std::max<int64_t>(max_group_rows * ns, 1);
    CU(c->d_cand.ensure(sizeof(double) * lm::kCandFields * p.cand_stride));
    p.cand = c->d_cand.as<double>();
  }
  std::vector<int> group_has_kernel(n_groups, 0);
  CU(c->d_nvalid.ensure(4 * (n_shard_nodes + 2)));
  CU(c->d_local_off.ensure(4 * (n_shard_nodes + 2)));
  CU(c->d_edge_off.ensure(4 * (n_shard_nodes + 2)));
  CU(c->d_edge_ng.ensure(4 * std::max<int64_t>(n_rows * ns, 1)));
  for (int g = 0; g < n_groups; ++g) {
    // blocks [bg0, bg1) with whole source images, views [gv0, gv1)
    const int bg1 = gb[g + 1];
    const int gv1 = (g + 1 < n_groups && bg1 < nb) ? blk[bg1].src_view : ve;
    const int64_t rb = row_off[bg0], re = row_off[bg1];
    const int64_t node_lo = c->line_off[gv0], node_hi = c->line_off[gv1];
    if (!exhaustive && re > rb) {
      int64_t need = 0;
      for (int b2 = bg0; b2 < bg1; ++b2) need = std::max(need, pair_off[b2] + blk[b2].n_rows);
      for (const auto &ch : c->chunks) // chunks complete in order: wait for the first one that covers `need`
        if (ch.row_end >= need) { CU(cudaStreamWaitEvent(sp, ch.ev, 0)); break; }
    }
    unsigned int *d_max_rows = c->d_scalars.as<unsigned int>() + 16 + g;
    if (row_sort_cub) {
      if (re > rb) {
        if (exhaustive)
          lm::launch_expand_exhaustive(c->d_blk_row_off.as<int64_t>(), c->d_blk_src.as<int32_t>(),
                                       c->d_blk_ng.as<int32_t>(), nb, c->d_line_off.as<int64_t>(), n_rows,
                                       c->d_key.as<uint32_t>(), c->d_val.as<uint32_t>(), sp);
        else
          lm::launch_expand_rows(c->d_pairs.as<int32_t>(), c->d_blk_row_off.as<int64_t>(), c->d_blk_src.as<int32_t>(),
                                 c->d_blk_ng.as<int32_t>(), c->d_blk_pair_off.as<int64_t>(), nb,
                                 c->d_line_off.as<int64_t>(), rb, re, c->d_key.as<uint32_t>(), c->d_val.as<uint32_t>(),
                                 d_err, sp);
        ++launches;
        CU(radix_sort_rows(rb, re));
      }
      lm::launch_node_offsets(c->sorted_key + rb, re - rb, rb, node_lo, node_hi, c->d_node_row_off.as<uint32_t>(),
                              d_max_rows, sp);
      ++launches;
    } else {
      const int i_lo = gv0 - vb, i_hi = gv1 - vb, n_tiles = vtile[i_hi] - vtile[i_lo];
      int max_lines = 0;
      for (int i = i_lo; i < i_hi; ++i) {
        const int64_t L = c->line_off[vb + i + 1] - c->line_off[vb + i];
        if (L <= lm::kRowSortMaxLines) max_lines = std::max(max_lines, (int)L);
      }
      CU(lm::launch_row_sort(c->d_pairs.as<int32_t>(), c->d_blk_row_off.as<int64_t>(), c->d_blk_ng.as<int32_t>(),
                             c->d_blk_pair_off.as<int64_t>(), nb, c->d_line_off.as<int64_t>(), vb,
                             c->d_rs_vrow.as<int64_t>(), c->d_rs_vtile.as<int32_t>(), c->d_rs_vtab.as<int64_t>(), i_lo,
                             i_hi, vtile[i_lo], n_tiles, max_lines, c->d_rs_tab.as<uint32_t>(),
                             c->d_node_row_off.as<uint32_t>(), d_max_rows, c->d_key2.as<uint32_t>(),
                             c->d_val2.as<uint32_t>(), d_err, sp));
      launches += (i_hi > i_lo) + (n_tiles > 0 ? 2 : 0);
      for (int i = i_lo; i < i_hi; ++i) { // views with too many lines for the shared-memory histograms
        const int64_t n0 = c->line_off[vb + i], n1 = c->line_off[vb + i + 1];
        if (n1 - n0 <= lm::kRowSortMaxLines) continue;
        const int64_t r0 = vrow[i], r1 = vrow[i + 1];
        if (r1 > r0) {
          lm::launch_expand_rows(c->d_pairs.as<int32_t>(), c->d_blk_row_off.as<int64_t>(), c->d_blk_src.as<int32_t>(),
                                 c->d_blk_ng.as<int32_t>(), c->d_blk_pair_off.as<int64_t>(), nb,
                                 c->d_line_off.as<int64_t>(), r0, r1, c->d_key.as<uint32_t>(), c->d_val.as<uint32_t>(),
                                 d_err, sp);
          ++launches;
          CU(radix_sort_rows(r0, r1));
        }
        lm::launch_node_offsets(c->sorted_key + r0, r1 - r0, r0, n0, n1, c->d_node_row_off.as<uint32_t>(), d_max_rows, sp);
        ++launches;
      }
    }
    CU(cudaEventRecord(c->evp[g], sp));
    CU(cudaStreamWaitEvent(s, c->evp[g], 0));
    p.node_begin = node_lo;
    p.node_end = node_hi;
    const int64_t n_group_nodes = node_hi - node_lo;
    size_t smem = split ? lm::tri_score_smem_bytes(cap_split) : lm::tri_smem_bytes(cap, fast_kernel);
    int grid;
    if (split) {
      p.use_slab = 0;
      p.cap = cap_split;
      p.row_begin = rb;
      p.row_end = re;
      grid = (int)std::min<int64_t>(n_group_nodes, (int64_t)1 << 30);
    } else if (smem <= smem_limit) {
      p.use_slab = 0;
      p.cap = cap;
      grid = (int)std::min<int64_t>(n_group_nodes, (int64_t)1 << 30);
    } else {
      // nodes larger than shared memory (exhaustive matching): persistent CTAs with a global staging slab
      p.use_slab = 1;
      p.cap = cap;
      grid = (int)std::min<int64_t>(n_group_nodes, (int64_t)c->sm_count * 4);
      p.slab_stride = (int64_t)((smem + 255) / 256 * 256);
      CU(c->d_slab.ensure((size_t)p.slab_stride * std::max(grid, 1)));
      p.slab = c->d_slab.as<char>();
      smem = 0;
    }
    if (n_group_nodes > 0) {
      CU(cudaEventRecord(c->evk[2 * g], s)); // node kernel time: generation through scoring
      if (split) CU(lm::launch_tri_split(p, grid, smem, s));
      else CU(lm::launch_tri_node_kernel(p, grid, 128, smem, s));
      CU(cudaEventRecord(c->evk[2 * g + 1], s));
      group_has_kernel[g] = 1;
      launches += split ? 2 : 1;
      // valid_edges_ of the group in compact form: per-node counts -> exclusive scan -> ordered scatter at the global
      // offsets
      {
        cudaStream_t so = c->out_stream; // under the node kernels of the later groups
        CU(cudaStreamWaitEvent(so, c->evk[2 * g + 1], 0));
        uint32_t *nv = c->d_nvalid.as<uint32_t>() + (node_lo - c->node_begin);
        lm::launch_extract_nvalid(p.nodes, node_lo, n_group_nodes, nv, so);
        size_t tmp = 0;
        CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, nv, c->d_local_off.as<uint32_t>(), (int)(n_group_nodes + 1), so));
        CU(c->d_scan_tmp.ensure(tmp)); // (not d_sort_tmp: the preparation stream sorts the next group meanwhile)
        CU(cub::DeviceScan::ExclusiveSum(c->d_scan_tmp.p, tmp, nv, c->d_local_off.as<uint32_t>(), (int)(n_group_nodes + 1), so));
        lm::launch_group_edges(p.row_state, p.row_ng, p.node_row_off, c->d_local_off.as<uint32_t>(),
                               c->d_scalars.as<unsigned int>() + 80, g, c->node_begin, node_lo, n_group_nodes, ns,
                               c->d_edge_off.as<uint32_t>(), c->d_edge_ng.as<uint32_t>(), so);
        launches += 4;
      }
      if (c->node_sink) { // the group's records go to the caller's buffer under the kernels of the later groups
        CU(cudaMemcpyAsync(c->node_sink + sizeof(lm::NodeRecord) * node_lo, c->d_nodes.as<lm::NodeRecord>() + node_lo,
                           sizeof(lm::NodeRecord) * n_group_nodes, cudaMemcpyDeviceToHost, c->out_stream));
      }
    }
    bg0 = bg1;
    gv0 = gv1;
  }
  p.node_begin = c->node_begin;
  p.node_end = c->node_end;
  CU(cudaGetLastError());
  // the engine's stream ends the run: whatever follows on it (getters, exchange) sees the compact connections
  CU(cudaEventRecord(c->ev_run_begin, c->out_stream));
  CU(cudaStreamWaitEvent(s, c->ev_run_begin, 0));
  CU(cudaEventRecord(c->ev1, s));
  // one read-back for the whole run: error / overflow flags, counters, largest node per group
  unsigned int *hs = c->h_pin;
  CU(cudaMemcpyAsync(hs, c->d_scalars.p, 512, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
#ifdef LM_TRACE
  fprintf(stderr, "[lm trace] compute stream drained %.3f ms after run entry\n", lm_ms());
#endif
  CU(cudaStreamSynchronize(c->copy_stream)); // uploads of images outside this shard may still be in flight
  CU(cudaStreamSynchronize(c->out_stream));
#ifdef LM_TRACE
  fprintf(stderr, "[lm trace] copy stream drained %.3f ms after run entry\n", lm_ms());
#endif
  c->stats.n_kernel_launches += launches;
  if (hs[1] == 1)
    return fail(LM_ERR_INVALID, "IndexError! Out-of-index matches exist (line_id >= number of lines of the image). "
                                "Please make sure you are reusing the correct descriptors and matches.");
  if (hs[1] == 2) return fail(LM_ERR_INVALID, "IndexError! Out-of-index neighbor line id in matches.");
  int max_rows_all = 0;
  for (int g = 0; g < n_groups; ++g) max_rows_all = std::max(max_rows_all, (int)hs[16 + g]);
  if ((int64_t)max_rows_all * ns > 65535) return fail(LM_ERR_INVALID, "more than 65535 candidates possible for one 2D line");
  int need_cap = 32;
  while (need_cap < max_rows_all * ns) need_cap += 32;
  c->cap_hint = need_cap;
  if (split) { // largest candidate count of a node in this run: the split scorer's capacity from now on
    int need_cand = 32;
    while (need_cand < (int)hs[3]) need_cand += 32;
    c->cap_hint_cand = need_cand;
  }
  if (hs[2] != 0) { // some node did not fit the staging area sized from the hint: repeat with the exact size
    if (c->run_retry) { c->run_retry = 0; return fail(LM_ERR_STATE, "node staging overflow after resizing"); }
    c->run_retry = 1;
    const int rc2 = lm_tri_run(c);
    c->run_retry = 0;
    return rc2;
  }
  float ms = 0;
  CU(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  for (int g = 0; g < n_groups; ++g)
    if (group_has_kernel[g]) {
      float msk = 0;
      CU(cudaEventElapsedTime(&msk, c->evk[2 * g], c->evk[2 * g + 1]));
      c->node_kernel_ms_acc += msk;
    }
  c->stats.max_rows_per_node = max_rows_all;
  c->stats.last_node_kernel_ms = c->node_kernel_ms_acc;
  const unsigned long long *cnt = reinterpret_cast<const unsigned long long *>(hs + 4);
  c->stats.n_rows = n_rows;
  c->stats.n_candidates = (int64_t)cnt[0];
  c->stats.n_valid_edges = (int64_t)cnt[1];
  c->stats.n_pairs_gated = (int64_t)cnt[2];
  c->stats.n_pairs_exact = (int64_t)cnt[3];
  c->stats.last_run_ms = ms;
  c->ran = true;
  return LM_OK;
}

int lm_tri_get_stats(lm_ctx *c, lm_tri_stats *out) {
  if (!c || !out) return fail(LM_ERR_INVALID, "NULL argument");
  *out = c->stats;
  return LM_OK;
}

int lm_tri_get_best(lm_ctx *c, int32_t img_id, double *out_line, int32_t *out_ng, int32_t *out_ncand) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  int rc = ensure_ran(c);
  if (rc) return rc;
  if ((rc = fetch_nodes(c))) return rc;
  auto it = c->id2view.find(img_id);
  if (it == c->id2view.end()) return fail(LM_ERR_INVALID, "unknown image id");
  const int v = it->second;
  for (int64_t n = c->line_off[v]; n < c->line_off[v + 1]; ++n) {
    const lm::NodeRecord &r = c->h_nodes[n];
    const int64_t l = n - c->line_off[v];
    for (int k = 0; k < 9; ++k) out_line[10 * l + k] = r.line[k];
    out_line[10 * l + 9] = r.score;
    out_ng[2 * l] = r.n_cand ? c->img_ids[r.ng_view] : 0;
    out_ng[2 * l + 1] = r.ng_line;
    if (out_ncand) out_ncand[l] = r.n_cand;
  }
  return LM_OK;
}

int64_t lm_tri_get_valid_edges(lm_ctx *c, int32_t img_id, int64_t *off, int32_t *edges) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  int rc = ensure_ran(c);
  if (rc) return rc;
  if ((rc = fetch_edges(c))) return rc;
  auto it = c->id2view.find(img_id);
  if (it == c->id2view.end()) return fail(LM_ERR_INVALID, "unknown image id");
  const int v = it->second;
  const int64_t L = c->line_off[v + 1] - c->line_off[v];
  const bool in_shard = c->line_off[v] >= c->node_begin && c->line_off[v + 1] <= c->node_end;
  int64_t n_out = 0;
  for (int64_t l = 0; l < L; ++l) {
    if (off) off[l] = n_out;
    if (!in_shard) continue;
    const int64_t i = c->line_off[v] + l - c->node_begin;
    for (uint32_t e = c->h_edge_off[i]; e < c->h_edge_off[i + 1]; ++e) {
      if (edges) {
        edges[2 * n_out] = c->img_ids[c->h_edge_ng[e] >> 16];
        edges[2 * n_out + 1] = (int32_t)(c->h_edge_ng[e] & 0xffffu);
      }
      ++n_out;
    }
  }
  if (off) off[L] = n_out;
  return n_out;
}

int lm_tri_get_cands_node(lm_ctx *c, int32_t img_id, int32_t line_id, int32_t cap, double *out_line, int32_t *out_ng) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (!c->have_cfg || !c->cfg.debug_mode) return fail(LM_ERR_STATE, "GetScoredTrisNode needs debug_mode");
  int rc = ensure_ran(c);
  if (rc) return rc;
  if ((rc = fetch_rows(c))) return rc;
  auto it = c->id2view.find(img_id);
  if (it == c->id2view.end()) return fail(LM_ERR_INVALID, "unknown image id");
  const int64_t n = c->line_off[it->second] + line_id;
  if (line_id < 0 || n >= c->line_off[it->second + 1]) return fail(LM_ERR_INVALID, "line id out of range");
  int k = 0;
  for (int64_t q = (int64_t)c->h_node_row_off[n] * c->ns; q < (int64_t)c->h_node_row_off[n + 1] * c->ns; ++q) {
    if (c->h_row_state[q] == 0) continue;
    const uint32_t r = (uint32_t)(q / c->ns);
    if (k < cap) {
      for (int t = 0; t < 10; ++t) out_line[10 * k + t] = c->h_row_cand[(size_t)q * 10 + t];
      out_ng[2 * k] = c->img_ids[c->h_row_ng[r] >> 16];
      out_ng[2 * k + 1] = (int32_t)(c->h_row_ng[r] & 0xffffu);
    }
    ++k;
  }
  return k;
}

int64_t lm_tri_num_nodes(lm_ctx *c) { return c ? c->n_nodes : 0; }
int64_t lm_scene_node_offset(lm_ctx *c, int32_t v) {
  if (!c || v < 0 || v > c->V) return -1;
  return c->line_off[v];
}
int lm_tri_export_nodes(lm_ctx *c, int64_t b, int64_t e, void *d_out) {
  if (!c || !d_out || b < 0 || e > c->n_nodes || b > e) return fail(LM_ERR_INVALID, "bad node range");
  int rc = ensure_ran(c);
  if (rc) return rc;
  CU(cudaMemcpyAsync(d_out, c->d_nodes.as<lm::NodeRecord>() + b, sizeof(lm::NodeRecord) * (e - b),
                     cudaMemcpyDeviceToDevice, c->stream));
  return LM_OK;
}
int lm_tri_import_nodes(lm_ctx *c, int64_t b, int64_t e, const void *d_in) {
  if (!c || !d_in || b < 0 || e > c->n_nodes || b > e) return fail(LM_ERR_INVALID, "bad node range");
  CU(c->d_nodes.ensure(sizeof(lm::NodeRecord) * std::max<int64_t>(c->n_nodes, 1)));
  CU(cudaMemcpyAsync(c->d_nodes.as<lm::NodeRecord>() + b, d_in, sizeof(lm::NodeRecord) * (e - b),
                     cudaMemcpyDeviceToDevice, c->stream));
  c->h_nodes_valid = false;
  return LM_OK;
}

static int collect_edges(lm_ctx *c) {
  if (c->edges_collected) {
    if (c->edges_count_on_device) {
      const int64_t over = lm_tri_gather_status(c, nullptr);
      if (over < 0) return (int)over;
      if (over) return fail(LM_ERR_STATE, "the last multi-GPU exchange overflowed its edge capacity: repeat it with a larger message");
    }
    return LM_OK;
  }
  const int64_t ne = c->stats.n_valid_edges;
  CU(c->d_edges.ensure(16 * std::max<int64_t>(ne, 1)));
  lm::launch_edge_pairs(c->d_edge_off.as<uint32_t>(), c->d_edge_ng.as<uint32_t>(), c->d_line_off.as<int64_t>(),
                        c->node_begin, c->node_end - c->node_begin, ne, c->d_edges.as<int64_t>(), c->stream);
  c->stats.n_kernel_launches += 1;
  c->n_edges_dev = ne;
  c->edges_collected = true;
  return LM_OK;
}
int64_t lm_tri_num_valid_edges(lm_ctx *c) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  int rc = ensure_ran(c);
  if (rc) return rc;
  if ((rc = collect_edges(c))) return rc;
  return c->n_edges_dev;
}
int lm_tri_export_edges(lm_ctx *c, void *d_out) {
  if (!c || !d_out) return fail(LM_ERR_INVALID, "NULL argument");
  int rc = ensure_ran(c);
  if (rc) return rc;
  if ((rc = collect_edges(c))) return rc;
  if (c->n_edges_dev)
    CU(cudaMemcpyAsync(d_out, c->d_edges.p, 16 * c->n_edges_dev, cudaMemcpyDeviceToDevice, c->stream));
  return LM_OK;
}
int lm_tri_import_edges(lm_ctx *c, int64_t n, const void *d_in, int32_t append) {
  if (!c || (n && !d_in)) return fail(LM_ERR_INVALID, "NULL argument");
  const int64_t base = append ? c->n_edges_dev : 0;
  if ((size_t)(base + n) * 16 > c->d_edges.cap) {
    DevBuf nb;
    CU(nb.ensure((size_t)(base + n) * 16));
    if (base) CU(cudaMemcpyAsync(nb.p, c->d_edges.p, 16 * base, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->d_edges.release();
    c->d_edges = nb;
  }
  if (n) CU(cudaMemcpyAsync(c->d_edges.as<char>() + 16 * base, d_in, 16 * n, cudaMemcpyDeviceToDevice, c->stream));
  c->n_edges_dev = base + n;
  c->edges_collected = true;
  return LM_OK;
}

int64_t lm_tri_gather_message_bytes(int64_t max_nodes, int64_t cap_edges) {
  if (max_nodes < 0 || cap_edges < 0) return fail(LM_ERR_INVALID, "bad sizes");
  return (16 + max_nodes * (int64_t)sizeof(lm::NodeRecord) + cap_edges * 8 + 15) / 16 * 16;
}
int lm_tri_pack_message(lm_ctx *c, int64_t max_nodes, int64_t cap_edges, void *d_msg) {
  if (!c || !d_msg) return fail(LM_ERR_INVALID, "NULL argument");
  int rc = ensure_ran(c);
  if (rc) return rc;
  const int64_t n = c->node_end - c->node_begin;
  if (n > max_nodes) return fail(LM_ERR_INVALID, "shard has more nodes than the message holds");
  lm::launch_gather_pack(c->d_nodes.as<lm::NodeRecord>(), c->node_begin, n, max_nodes, c->d_edge_off.as<uint32_t>(),
                         c->d_edge_ng.as<uint32_t>(), c->d_line_off.as<int64_t>(), cap_edges, static_cast<char *>(d_msg),
                         c->stream);
  CU(cudaGetLastError());
  c->stats.n_kernel_launches += 1;
  return LM_OK;
}
int lm_tri_unpack_messages(lm_ctx *c, int32_t world, const int64_t *rank_node_begin, int64_t max_nodes, int64_t cap_edges,
                           const void *d_msgs) {
  if (!c || !d_msgs || !rank_node_begin || world <= 0 || world > 64) return fail(LM_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  for (int r = 0; r < world; ++r)
    if (rank_node_begin[r] < 0 || rank_node_begin[r] > c->n_nodes) return fail(LM_ERR_INVALID, "bad node range");
  CU(c->d_nodes.ensure(sizeof(lm::NodeRecord) * std::max<int64_t>(c->n_nodes, 1)));
  if ((size_t)world * cap_edges * 16 + 16 > c->d_edges.cap) {
    CU(cudaStreamSynchronize(c->stream));
    CU(c->d_edges.ensure((size_t)world * cap_edges * 16 + 16));
  }
  CU(c->d_gather.ensure(8 * 64 + 64));
  // rank table as kernel-readable memory: tiny, written through pinned memory on the compute stream's own order
  int64_t *h = reinterpret_cast<int64_t *>(c->h_pin + 128); // bytes 512.. of the pinned pad
  for (int r = 0; r < world; ++r) h[r] = rank_node_begin[r];
  if (memcmp(c->gather_tab, h, 8 * world) != 0 || c->gather_world != world) {
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpyAsync(c->d_gather.as<char>() + 64, h, 8 * world, cudaMemcpyHostToDevice, c->copy_stream));
    CU(cudaStreamSynchronize(c->copy_stream));
    memcpy(c->gather_tab, h, 8 * world);
    c->gather_world = world;
  }
  lm::launch_gather_unpack(static_cast<const char *>(d_msgs), world, reinterpret_cast<const int64_t *>(c->d_gather.as<char>() + 64),
                           max_nodes, cap_edges, lm_tri_gather_message_bytes(max_nodes, cap_edges),
                           c->d_nodes.as<lm::NodeRecord>(), c->d_edges.as<int64_t>(), c->d_gather.as<int64_t>(), c->stream);
  CU(cudaGetLastError());
  c->stats.n_kernel_launches += 1;
  c->h_nodes_valid = false;
  c->edges_collected = true;
  c->edges_count_on_device = true;
  return LM_OK;
}
int64_t lm_tri_gather_status(lm_ctx *c, int64_t *n_edges_total) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  if (!c->edges_count_on_device) { if (n_edges_total) *n_edges_total = c->n_edges_dev; return 0; }
  int64_t *h = reinterpret_cast<int64_t *>(c->h_pin + 256);
  CU(cudaMemcpyAsync(h, c->d_gather.p, 16, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  c->n_edges_dev = h[0];
  c->edges_count_on_device = false;
  if (n_edges_total) *n_edges_total = h[0];
  return h[1]; // 1: some rank had more valid connections than cap_edges -- repeat the exchange with a larger message
}

// ---- ComputeLineTracks ---------------------------------------------------------------------------
namespace {

// Symmetric 3x3 Jacobi eigen-solver (dominant eigenvector) for the total-least-squares direction of
// Aggregator::aggregate_line3d_list (merging/aggregator.cc:63-78; JacobiSVD V.col(0) up to sign).
void dominant_eigvec(const double Ain[3][3], double out[3]) {
  double A[3][3], V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  memcpy(A, Ain, sizeof(A));
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = A[0][1] * A[0][1] + A[0][2] * A[0][2] + A[1][2] * A[1][2];
    double diag = A[0][0] * A[0][0] + A[1][1] * A[1][1] + A[2][2] * A[2][2];
    if (off == 0 || off <= 1e-32 * diag) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (A[p][q] == 0) continue;
        double theta = (A[q][q] - A[p][p]) / (2 * A[p][q]);
        double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1));
        double cs = 1 / std::sqrt(t * t + 1), sn = t * cs;
        for (int k = 0; k < 3; ++k) { double a = A[k][p], b = A[k][q]; A[k][p] = cs * a - sn * b; A[k][q] = sn * a + cs * b; }
        for (int k = 0; k < 3; ++k) { double a = A[p][k], b = A[q][k]; A[p][k] = cs * a - sn * b; A[q][k] = sn * a + cs * b; }
        for (int k = 0; k < 3; ++k) { double a = V[k][p], b = V[k][q]; V[k][p] = cs * a - sn * b; V[k][q] = sn * a + cs * b; }
      }
  }
  int best = 0;
  if (A[1][1] > A[best][best]) best = 1;
  if (A[2][2] > A[best][best]) best = 2;
  for (int k = 0; k < 3; ++k) out[k] = V[k][best];
}

struct AggItem { // one Line3d of a line3d_list: endpoints, uncertainty, score
  const double *l;
  double unc, score;
};
void aggregate_items(const std::vector<AggItem> &it, int num_outliers, double out[7]) {
  const int n = (int)it.size();
  double min_unc = 1.7976931348623157e308;
  for (const AggItem &r : it) if (r.unc < min_unc) min_unc = r.unc;
  if (n < 4) { // aggregate_line3d_list_takebest (aggregator.cc:9-29); index 0 when no score > 0
    double best_score = 0.0;
    int best = -1;
    for (int i = 0; i < n; ++i) if (it[i].score > best_score) { best_score = it[i].score; best = i; }
    if (best < 0) best = 0;
    for (int k = 0; k < 6; ++k) out[k] = it[best].l[k];
    out[6] = min_unc;
    return;
  }
  double ctr[3] = {0, 0, 0};
  for (const AggItem &r : it) for (int k = 0; k < 3; ++k) { ctr[k] += r.l[k]; ctr[k] += r.l[3 + k]; }
  for (int k = 0; k < 3; ++k) ctr[k] = ctr[k] / (2 * n);
  double S[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
  for (const AggItem &r : it)
    for (int e = 0; e < 2; ++e) {
      double p[3] = {r.l[3 * e] - ctr[0], r.l[3 * e + 1] - ctr[1], r.l[3 * e + 2] - ctr[2]};
      for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) S[a][b] += p[a] * p[b];
    }
  double d[3];
  dominant_eigvec(S, d);
  double dn = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
  for (int k = 0; k < 3; ++k) d[k] /= dn;
  std::vector<double> proj;
  for (const AggItem &r : it)
    for (int e = 0; e < 2; ++e)
      proj.push_back((r.l[3 * e] - ctr[0]) * d[0] + (r.l[3 * e + 1] - ctr[1]) * d[1] + (r.l[3 * e + 2] - ctr[2]) * d[2]);
  std::sort(proj.begin(), proj.end());
  const double a = proj[num_outliers], b = proj[2 * n - 1 - num_outliers];
  for (int k = 0; k < 3; ++k) { out[k] = ctr[k] + d[k] * a; out[3 + k] = ctr[k] + d[k] * b; }
  out[6] = min_unc;
}
void aggregate(const std::vector<const lm::NodeRecord *> &recs, int num_outliers, double out[7]) {
  std::vector<AggItem> it(recs.size());
  for (size_t i = 0; i < recs.size(); ++i) it[i] = AggItem{recs[i]->line, recs[i]->line[8], recs[i]->score};
  aggregate_items(it, num_outliers, out);
}

size_t uf_root(size_t i, std::vector<int> &parent) { // base/graph.cc:157-166
  size_t r = i;
  while (parent[r] != -1) r = parent[r];
  while (parent[i] != -1) { size_t nx = parent[i]; parent[i] = (int)r; i = nx; } // full compression to the root
  return r;
}

} // namespace

// The track graph on the device (graph_kernels.cu): from the directed valid connections in c->d_edges to the graph nodes
// in FindOrCreateNode order and the edges in the order ComputeLineTrackLabelsGreedy visits them, each edge as
// (idx0 << 32 | idx1). Two small read-backs; the union-find that follows is sequential by definition.
static int graph_on_device(lm_ctx *c, int64_t ne, std::vector<int64_t> &gnode, std::vector<uint64_t> &order) {
  cudaStream_t s = c->stream;
  gnode.clear();
  order.clear();
  if (ne <= 0) return LM_OK;
  if (ne >= (int64_t)1 << 30) return fail(LM_ERR_INVALID, "too many valid connections for the 32-bit positions of the graph build");
  auto sort_keys = [&](DevBuf &a, DevBuf &b, int64_t n, uint64_t *&out) -> int {
    cub::DoubleBuffer<uint64_t> dk(a.as<uint64_t>(), b.as<uint64_t>());
    size_t tmp = 0;
    CU(cub::DeviceRadixSort::SortKeys(nullptr, tmp, dk, (int)n, 0, 64, s));
    CU(c->d_sort_tmp.ensure(tmp));
    CU(cub::DeviceRadixSort::SortKeys(c->d_sort_tmp.p, tmp, dk, (int)n, 0, 64, s));
    out = dk.Current();
    return LM_OK;
  };
  auto scan_u32 = [&](const uint32_t *in, uint32_t *out, int64_t n) -> int {
    size_t tmp = 0;
    CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, (int)n, s));
    CU(c->d_sort_tmp.ensure(tmp));
    CU(cub::DeviceScan::ExclusiveSum(c->d_sort_tmp.p, tmp, in, out, (int)n, s));
    return LM_OK;
  };
  int rc;
  // undirected edge set in std::set order (:243-261)
  CU(c->d_edge_keys.ensure(8 * ne));
  CU(c->d_edge_keys2.ensure(8 * ne + 8));
  lm::launch_undirected_keys(c->d_edges.as<int64_t>(), ne, c->d_edge_keys.as<uint64_t>(), s);
  uint64_t *sorted = nullptr;
  if ((rc = sort_keys(c->d_edge_keys, c->d_edge_keys2, ne, sorted))) return rc;
  uint64_t *ukeys = (sorted == c->d_edge_keys.as<uint64_t>()) ? c->d_edge_keys2.as<uint64_t>() : c->d_edge_keys.as<uint64_t>();
  CU(c->d_edge_cnt.ensure(16));
  {
    size_t tmp = 0;
    CU(cub::DeviceSelect::Unique(nullptr, tmp, sorted, ukeys, c->d_edge_cnt.as<int64_t>(), (int)ne, s));
    CU(c->d_sort_tmp.ensure(tmp));
    CU(cub::DeviceSelect::Unique(c->d_sort_tmp.p, tmp, sorted, ukeys, c->d_edge_cnt.as<int64_t>(), (int)ne, s));
  }
  int64_t nu = 0;
  CU(cudaMemcpyAsync(&nu, c->d_edge_cnt.p, 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  // 3d score of every undirected edge (:263-288)
  CU(c->d_edges2.ensure(16 * nu));
  CU(c->d_edge_w.ensure(8 * nu));
  lm::launch_keys_to_pairs(ukeys, nu, c->d_edges2.as<int64_t>(), s);
  lm::EdgeParams ep;
  ep.nodes = c->d_nodes.as<lm::NodeRecord>();
  ep.edges = c->d_edges2.as<int64_t>();
  ep.weight = c->d_edge_w.as<double>();
  ep.n = nu;
  {
    lm_linker_config l3 = c->cfg.linker3d; // set_to_spatial_merging (line_linker.h:123-129)
    l3.use_angle = 1; l3.use_overlap = 1; l3.use_perp = 0; l3.use_innerseg = 1; l3.use_scaleinv = 0;
    ep.l3d = to_dev<double>(l3);
  }
  lm::launch_edge_weights(ep, s);
  // zero-score edges dropped, order kept (:284-285)
  CU(c->d_g_flag.ensure(4 * (2 * nu + 2)));
  CU(c->d_g_pos.ensure(4 * (2 * nu + 2)));
  CU(c->d_g_kc.ensure(8 * nu + 8));
  CU(c->d_g_wc.ensure(8 * nu + 8));
  uint32_t *flag = c->d_g_flag.as<uint32_t>(), *pos = c->d_g_pos.as<uint32_t>();
  lm::launch_nonzero_flags(c->d_edge_w.as<double>(), nu, flag, s);
  CU(cudaMemsetAsync(flag + nu, 0, 4, s)); // the scan of n + 1 flags ends with the total
  if ((rc = scan_u32(flag, pos, nu + 1))) return rc;
  lm::launch_compact_weighted_edges(ukeys, c->d_edge_w.as<double>(), flag, pos, nu, c->d_g_kc.as<uint64_t>(),
                                    c->d_g_wc.as<double>(), s);
  uint32_t n2u = 0;
  CU(cudaMemcpyAsync(&n2u, pos + nu, 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  const int64_t n2 = n2u;
  c->stats.n_kernel_launches += 12;
  if (n2 == 0) return LM_OK;
  // Graph::FindOrCreateNode numbering: rank of a node's first appearance in u0 v0 u1 v1 ...
  const int64_t m = 2 * n2;
  CU(c->d_g_occ.ensure(8 * m));
  CU(c->d_g_occ2.ensure(8 * m));
  lm::launch_occurrence_keys(c->d_g_kc.as<uint64_t>(), n2, c->d_g_occ.as<uint64_t>(), s);
  uint64_t *occ = nullptr;
  if ((rc = sort_keys(c->d_g_occ, c->d_g_occ2, m, occ))) return rc;
  lm::launch_occurrence_heads(occ, m, flag, s);
  CU(cudaMemsetAsync(flag + m, 0, 4, s));
  if ((rc = scan_u32(flag, pos, m + 1))) return rc;
  uint32_t ngu = 0;
  CU(cudaMemcpyAsync(&ngu, pos + m, 4, cudaMemcpyDeviceToHost, s));
  CU(c->d_g_hk.ensure(8 * m));
  CU(c->d_g_hk2.ensure(8 * m));
  lm::launch_head_keys(occ, flag, pos, m, c->d_g_hk.as<uint64_t>(), s);
  CU(cudaStreamSynchronize(s));
  const int64_t ng = ngu;
  uint64_t *hk = nullptr;
  if ((rc = sort_keys(c->d_g_hk, c->d_g_hk2, ng, hk))) return rc;
  CU(c->d_g_gidx.ensure(4 * (size_t)std::max<int64_t>(c->n_nodes, 1)));
  CU(c->d_g_gnode.ensure(4 * ng));
  lm::launch_graph_index(hk, ng, c->d_g_gidx.as<int32_t>(), c->d_g_gnode.as<int32_t>(), s);
  // edges in descending (score, idx0, idx1) order: stable LSD, nodes first, score second
  CU(c->d_g_k1.ensure(8 * n2)); CU(c->d_g_k1b.ensure(8 * n2));
  CU(c->d_g_k2.ensure(8 * n2)); CU(c->d_g_k2b.ensure(8 * n2));
  lm::launch_edge_order_keys(c->d_g_kc.as<uint64_t>(), c->d_g_wc.as<double>(), c->d_g_gidx.as<int32_t>(), n2,
                             c->d_g_k1.as<uint64_t>(), c->d_g_k2.as<uint64_t>(), s);
  const uint64_t *final_nodes = nullptr;
  {
    cub::DoubleBuffer<uint64_t> k(c->d_g_k1.as<uint64_t>(), c->d_g_k1b.as<uint64_t>());
    cub::DoubleBuffer<uint64_t> v(c->d_g_k2.as<uint64_t>(), c->d_g_k2b.as<uint64_t>());
    size_t tmp = 0;
    CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp, k, v, (int)n2, 0, 64, s));
    CU(c->d_sort_tmp.ensure(tmp));
    CU(cub::DeviceRadixSort::SortPairs(c->d_sort_tmp.p, tmp, k, v, (int)n2, 0, 64, s)); // by (idx0, idx1), scores carried
    cub::DoubleBuffer<uint64_t> k2(v.Current(), v.Alternate());
    cub::DoubleBuffer<uint64_t> v2(k.Current(), k.Alternate());
    size_t tmp2 = 0;
    CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp2, k2, v2, (int)n2, 0, 64, s));
    CU(c->d_sort_tmp.ensure(tmp2));
    CU(cub::DeviceRadixSort::SortPairs(c->d_sort_tmp.p, tmp2, k2, v2, (int)n2, 0, 64, s)); // by score, stable
    final_nodes = v2.Current();
  }
  std::vector<int32_t> gn32((size_t)ng);
  order.resize((size_t)n2);
  CU(cudaMemcpyAsync(gn32.data(), c->d_g_gnode.p, 4 * ng, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(order.data(), final_nodes, 8 * n2, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  c->stats.n_kernel_launches += 16;
  gnode.assign(gn32.begin(), gn32.end());
  for (uint64_t &o : order) o = ~o;
  return LM_OK;
}

int64_t lm_tri_build_tracks(lm_ctx *c, int64_t *n_support_total) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  int rc = ensure_ran(c);
  if (rc) return rc;
  CU(cudaSetDevice(c->device));
  if ((rc = collect_edges(c))) return rc;
  if ((rc = fetch_nodes(c))) return rc;
  cudaStream_t s = c->stream;
  const int64_t ne = c->n_edges_dev;
  static const bool trace = getenv("LIMAP_B200_TRACE") != nullptr;
  const auto tr0 = std::chrono::steady_clock::now();
  auto tr_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tr0).count(); };
  c->tracks.clear();
  c->graph_nodes.clear();
  if (n_support_total) *n_support_total = 0;
  if (ne == 0) return 0;
  std::vector<int64_t> gnode;
  std::vector<uint64_t> order; // (idx0 << 32 | idx1) of every graph edge, in the order the greedy labelling visits them
  if (c->cfg.min_num_outer_edges <= 0) {
    // (filterNodeByNumOuterEdges keeps every node: the whole graph is built on the device)
    if ((rc = graph_on_device(c, ne, gnode, order))) return rc;
  } else {
  std::vector<int64_t> h_edges(2 * ne);
  CU(cudaMemcpyAsync(h_edges.data(), c->d_edges.p, 16 * ne, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));

  // filterNodeByNumOuterEdges (global_line_triangulator.cc:168-232)
  std::vector<char> flag(c->n_nodes, 1);
  const int min_outer = c->cfg.min_num_outer_edges;
  if (min_outer > 0) {
    std::vector<int> counter(c->n_nodes, 0);
    std::vector<int64_t> pstart(c->n_nodes + 1, 0);
    for (int64_t e = 0; e < ne; ++e) { counter[h_edges[2 * e]]++; pstart[h_edges[2 * e + 1] + 1]++; }
    for (int64_t n = 0; n < c->n_nodes; ++n) pstart[n + 1] += pstart[n];
    std::vector<int64_t> parents(ne), fill(pstart.begin(), pstart.end() - 1);
    for (int64_t e = 0; e < ne; ++e) parents[fill[h_edges[2 * e + 1]]++] = h_edges[2 * e];
    std::queue<int64_t> q;
    for (int64_t n = 0; n < c->n_nodes; ++n)
      if (counter[n] < min_outer) { flag[n] = 0; q.push(n); }
    while (!q.empty()) {
      int64_t n = q.front(); q.pop();
      for (int64_t k = pstart[n]; k < pstart[n + 1]; ++k) {
        int64_t pn = parents[k];
        if (!flag[pn]) continue;
        if (--counter[pn] < min_outer) { flag[pn] = 0; q.push(pn); }
      }
    }
  }
  // undirected edge set ordered like std::set<pair<LineNode,LineNode>> (:243-261): sort + unique on device
  std::vector<uint64_t> keys;
  keys.reserve(ne);
  for (int64_t e = 0; e < ne; ++e) {
    int64_t a = h_edges[2 * e], b = h_edges[2 * e + 1];
    if (!flag[a] || !flag[b]) continue;
    if (a > b) std::swap(a, b);
    keys.push_back(((uint64_t)a << 32) | (uint64_t)b);
  }
  const int64_t nk = (int64_t)keys.size();
  if (nk == 0) return 0;
  CU(c->d_edge_keys.ensure(8 * nk));
  CU(c->d_edge_keys2.ensure(8 * nk + 8));
  CU(cudaMemcpyAsync(c->d_edge_keys.p, keys.data(), 8 * nk, cudaMemcpyHostToDevice, s));
  {
    cub::DoubleBuffer<uint64_t> dk(c->d_edge_keys.as<uint64_t>(), c->d_edge_keys2.as<uint64_t>());
    size_t tmp = 0;
    CU(cub::DeviceRadixSort::SortKeys(nullptr, tmp, dk, (int)nk, 0, 64, s));
    CU(c->d_sort_tmp.ensure(tmp));
    CU(cub::DeviceRadixSort::SortKeys(c->d_sort_tmp.p, tmp, dk, (int)nk, 0, 64, s));
    uint64_t *sorted = dk.Current();
    uint64_t *other = dk.Alternate();
    size_t tmp2 = 0;
    CU(c->d_edge_cnt.ensure(8));
    CU(cub::DeviceSelect::Unique(nullptr, tmp2, sorted, other, c->d_edge_cnt.as<int64_t>(), (int)nk, s));
    CU(c->d_sort_tmp.ensure(tmp2));
    CU(cub::DeviceSelect::Unique(c->d_sort_tmp.p, tmp2, sorted, other, c->d_edge_cnt.as<int64_t>(), (int)nk, s));
    int64_t nu = 0;
    CU(cudaMemcpyAsync(&nu, c->d_edge_cnt.p, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    keys.resize(nu);
    CU(cudaMemcpyAsync(keys.data(), other, 8 * nu, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    c->stats.n_kernel_launches += 12;
  }
  const int64_t nu = (int64_t)keys.size();
  // 3d score of every undirected edge on the device (:263-288)
  std::vector<int64_t> ue(2 * nu);
  for (int64_t e = 0; e < nu; ++e) { ue[2 * e] = (int64_t)(keys[e] >> 32); ue[2 * e + 1] = (int64_t)(keys[e] & 0xffffffffull); }
  CU(c->d_edges2.ensure(16 * nu));
  CU(c->d_edge_w.ensure(8 * nu));
  CU(cudaMemcpyAsync(c->d_edges2.p, ue.data(), 16 * nu, cudaMemcpyHostToDevice, s));
  lm::EdgeParams ep;
  ep.nodes = c->d_nodes.as<lm::NodeRecord>();
  ep.edges = c->d_edges2.as<int64_t>();
  ep.weight = c->d_edge_w.as<double>();
  ep.n = nu;
  {
    lm_linker_config l3 = c->cfg.linker3d; // set_to_spatial_merging (line_linker.h:123-129)
    l3.use_angle = 1; l3.use_overlap = 1; l3.use_perp = 0; l3.use_innerseg = 1; l3.use_scaleinv = 0;
    ep.l3d = to_dev<double>(l3);
  }
  lm::launch_edge_weights(ep, s);
  c->stats.n_kernel_launches += 1;
  std::vector<double> w(nu);
  CU(cudaMemcpyAsync(w.data(), c->d_edge_w.p, 8 * nu, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));

  // Graph::FindOrCreateNode in edge order (base/graph.cc:57-70), zero-score edges dropped first (:284-285)
  std::unordered_map<int64_t, int> node_map;
  typedef std::tuple<double, size_t, size_t> edge_tuple;
  std::vector<edge_tuple> edges;
  for (int64_t e = 0; e < nu; ++e) {
    if (w[e] == 0) continue;
    size_t idx[2];
    for (int k = 0; k < 2; ++k) {
      auto f = node_map.find(ue[2 * e + k]);
      if (f == node_map.end()) {
        gnode.push_back(ue[2 * e + k]);
        idx[k] = gnode.size() - 1;
        node_map.emplace(ue[2 * e + k], (int)idx[k]);
      } else
        idx[k] = f->second;
    }
    edges.push_back(std::make_tuple(w[e], idx[0], idx[1]));
  }
  // ComputeLineTrackLabelsGreedy (merging/merging.cc:18-103): edges by descending (score, node, node)
  std::sort(edges.begin(), edges.end());
  std::reverse(edges.begin(), edges.end());
  order.reserve(edges.size());
  for (const edge_tuple &e : edges) order.push_back((uint64_t)std::get<1>(e) << 32 | (uint64_t)std::get<2>(e));
  } // host graph (min_num_outer_edges > 0)
  const size_t n_gn = gnode.size();
  if (trace) fprintf(stderr, "[lm trace] build_tracks: graph (%zu nodes, %zu edges) ready at %.2f ms\n", n_gn, order.size(), tr_ms());
  if (n_gn == 0) return 0;
  std::vector<int> parent(n_gn, -1);
  // view index of a graph node: binary search in line_off
  std::vector<int> view_of(n_gn);
  for (size_t i = 0; i < n_gn; ++i)
    view_of[i] = (int)(std::upper_bound(c->line_off.begin(), c->line_off.end(), gnode[i]) - c->line_off.begin()) - 1;
  // The reference's union_find_get_root compresses recursively (every node on the path points to the
  // root afterwards); uf_root does the same iteratively. The union direction depends on the number of DISTINCT images
  // of the two tracks (merging.cc:40-50): a bit set per root when the scene has few views (a union is an OR and a
  // popcount), sorted id vectors otherwise.
  const int V = c->V;
  const char *bs_env = getenv("LIMAP_B200_UF_BITSET_MAX_VIEWS"); // (tests force the vector path with 0)
  if (V <= (bs_env ? atoi(bs_env) : 1024)) {
    const size_t W = (size_t)(V + 63) / 64;
    std::vector<uint64_t> bits(n_gn * W, 0);
    std::vector<int> n_img(n_gn, 1);
    for (size_t i = 0; i < n_gn; ++i) bits[i * W + (size_t)view_of[i] / 64] = 1ull << (view_of[i] % 64);
    for (const uint64_t e : order) {
      size_t r1 = uf_root((size_t)(e >> 32), parent), r2 = uf_root((size_t)(e & 0xffffffffull), parent);
      if (r1 == r2) continue;
      size_t dst, srcn;
      if (n_img[r1] < n_img[r2]) { parent[r1] = (int)r2; dst = r2; srcn = r1; }
      else { parent[r2] = (int)r1; dst = r1; srcn = r2; }
      int cnt = 0;
      for (size_t w = 0; w < W; ++w) {
        bits[dst * W + w] |= bits[srcn * W + w];
        cnt += __builtin_popcountll(bits[dst * W + w]);
      }
      n_img[dst] = cnt;
    }
  } else {
    std::vector<std::vector<int>> images(n_gn); // sorted distinct image ids of each root's track
    for (size_t i = 0; i < n_gn; ++i) images[i].push_back(view_of[i]);
    for (const uint64_t e : order) {
      size_t r1 = uf_root((size_t)(e >> 32), parent), r2 = uf_root((size_t)(e & 0xffffffffull), parent);
      if (r1 == r2) continue;
      size_t dst, srcn;
      if (images[r1].size() < images[r2].size()) { parent[r1] = (int)r2; dst = r2; srcn = r1; }
      else { parent[r2] = (int)r1; dst = r1; srcn = r2; }
      std::vector<int> merged;
      std::set_union(images[dst].begin(), images[dst].end(), images[srcn].begin(), images[srcn].end(),
                     std::back_inserter(merged));
      images[dst].swap(merged);
      std::vector<int>().swap(images[srcn]);
    }
  }
  if (trace) fprintf(stderr, "[lm trace] build_tracks: union-find done at %.2f ms\n", tr_ms());
  std::vector<int> label(n_gn, -1);
  int n_tracks = 0;
  for (size_t i = 0; i < n_gn; ++i) {
    if (parent[i] == -1) continue;
    size_t pi = parent[i];
    if (parent[pi] == -1 && label[pi] == -1) label[pi] = n_tracks++;
  }
  for (size_t i = 0; i < n_gn; ++i) {
    if (parent[i] == -1) continue;
    label[i] = label[uf_root(i, parent)];
  }
  // build_tracks_from_clusters (global_line_triangulator.cc:293-351)
  c->tracks.assign(n_tracks, Track());
  int64_t support = 0;
  for (size_t i = 0; i < n_gn; ++i) {
    if (label[i] < 0) continue;
    Track &t = c->tracks[label[i]];
    const int v = view_of[i];
    t.img.push_back(c->img_ids[v]);
    t.line.push_back((int)(gnode[i] - c->line_off[v]));
    t.node.push_back((int)i);
    t.gid.push_back(gnode[i]);
    ++support;
  }
  for (Track &t : c->tracks) {
    std::vector<const lm::NodeRecord *> recs;
    for (int64_t g : t.gid) recs.push_back(&c->h_nodes[g]);
    aggregate(recs, c->cfg.num_outliers_aggregator, t.agg);
  }
  c->graph_nodes.clear();
  if (n_support_total) *n_support_total = support;
  if (trace) fprintf(stderr, "[lm trace] build_tracks: %d tracks aggregated at %.2f ms\n", n_tracks, tr_ms());
  return n_tracks;
}

int lm_tri_get_tracks(lm_ctx *c, int64_t *track_off, int32_t *img_ids, int32_t *line_ids, int32_t *node_ids,
                      double *node_line3d, double *track_line) {
  if (!c) return fail(LM_ERR_INVALID, "ctx is NULL");
  int64_t n = 0;
  for (size_t t = 0; t < c->tracks.size(); ++t) {
    const Track &tr = c->tracks[t];
    track_off[t] = n;
    for (size_t k = 0; k < tr.img.size(); ++k, ++n) {
      img_ids[n] = tr.img[k];
      line_ids[n] = tr.line[k];
      node_ids[n] = tr.node[k];
      const lm::NodeRecord &r = c->h_nodes[tr.gid[k]];
      for (int q = 0; q < 9; ++q) node_line3d[10 * n + q] = r.line[q];
      node_line3d[10 * n + 9] = r.score;
    }
    for (int q = 0; q < 7; ++q) track_line[7 * t + q] = tr.agg[q];
  }
  track_off[c->tracks.size()] = n;
  return LM_OK;
}

} // extern "C"

// ---- line refinement ------------------------------------------------------------------------------
namespace {

struct V3h { double x, y, z; };
inline V3h v3(double x, double y, double z) { return V3h{x, y, z}; }
inline V3h crossh(V3h a, V3h b) { return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }

// MinimalInfiniteLine3d::GetInfiniteLine (:220-231) + GetLineSegmentFromInfiniteLine3d (:265-287)
void segment_from_minimal(const double x[6], const double *l3d, int64_t n, int num_outliers, double out[6]) {
  M3h Q = quat_to_R(x);
  const V3h d = v3(Q.m[0], Q.m[3], Q.m[6]);
  const double f = std::fabs(x[5]) / std::fabs(x[4]);
  const V3h m = v3(Q.m[1] * f, Q.m[4] * f, Q.m[7] * f);
  auto point_projection = [&](V3h q) { // InfiniteLine3d::point_projection (:73-78)
    V3h dq = crossh(d, q);
    V3h mq = v3(m.x + dq.x, m.y + dq.y, m.z + dq.z);
    V3h c = crossh(d, mq);
    return v3(q.x + c.x, q.y + c.y, q.z + c.z);
  };
  const V3h pref = point_projection(v3(l3d[0], l3d[1], l3d[2]));
  std::vector<double> vals;
  vals.reserve(2 * n);
  for (int64_t k = 0; k < n; ++k)
    for (int e = 0; e < 2; ++e) {
      const double *p = l3d + 6 * k + 3 * e;
      vals.push_back((p[0] - pref.x) * d.x + (p[1] - pref.y) * d.y + (p[2] - pref.z) * d.z);
    }
  std::sort(vals.begin(), vals.end());
  const double a = vals[num_outliers], b = vals[2 * n - 1 - num_outliers];
  out[0] = pref.x + d.x * a; out[1] = pref.y + d.y * a; out[2] = pref.z + d.z * a;
  out[3] = pref.x + d.x * b; out[4] = pref.y + d.y * b; out[5] = pref.z + d.z * b;
}

} // namespace

extern "C" {

int lm_ba_solve(lm_ctx *c, int32_t n_views, const double *kvec, const double *qvec, const double *tvec, int64_t T,
                const int64_t *sup_off, const int32_t *sup_view, const double *segs, const double *line3d,
                const double *line_init, const double *sup_vp, const lm_ba_config *cfg, double *out_line,
                double *out_minimal, int32_t *out_iters, double *out_cost) {
  if (!c || !cfg || !sup_off) return fail(LM_ERR_INVALID, "NULL argument");
  if (T < 0 || n_views <= 0) return fail(LM_ERR_INVALID, "bad sizes");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const int64_t n = sup_off[T];
  for (int64_t k = 0; k < n; ++k)
    if (sup_view[k] < 0 || sup_view[k] >= n_views) return fail(LM_ERR_INVALID, "support view index out of range");
  // device input arena: [kvec | qvec | tvec | segs | x0 | sup_off | sup_view | active]
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const size_t o_k = take(32 * n_views), o_q = take(32 * n_views), o_t = take(24 * n_views), o_s = take(32 * n),
               o_x = take(48 * T), o_so = take(8 * (T + 1)), o_sv = take(4 * n), o_a = take(T),
               o_vp = take(sup_vp ? 24 * n : 0), o_l3 = take((line3d && out_line) ? 48 * n : 0), o_li = take(48 * T),
               o_err = take(32);
  CU(c->d_ba_in.ensure(off + 256));
  char *in = c->d_ba_in.as<char>();
  CU(cudaMemcpyAsync(in + o_k, kvec, 32 * n_views, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_q, qvec, 32 * n_views, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_t, tvec, 24 * n_views, cudaMemcpyHostToDevice, s));
  if (n) CU(cudaMemcpyAsync(in + o_s, segs, 32 * n, cudaMemcpyHostToDevice, s));
  if (T) CU(cudaMemcpyAsync(in + o_li, line_init, 48 * T, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_so, sup_off, 8 * (T + 1), cudaMemcpyHostToDevice, s));
  if (n) CU(cudaMemcpyAsync(in + o_sv, sup_view, 4 * n, cudaMemcpyHostToDevice, s));
  if (sup_vp && n) CU(cudaMemcpyAsync(in + o_vp, sup_vp, 24 * n, cudaMemcpyHostToDevice, s));
  const bool dev_seg = line3d && out_line && n;
  if (dev_seg) CU(cudaMemcpyAsync(in + o_l3, line3d, 48 * n, cudaMemcpyHostToDevice, s));
  CU(c->d_ba_blocks.ensure(sizeof(lm::LMBlockDev) * std::max<int64_t>(n, 1)));
  size_t oo = 0;
  auto take_o = [&](size_t bytes) { size_t o = oo; oo += (bytes + 255) / 256 * 256; return o; };
  const size_t oo_x = take_o(48 * T), oo_i = take_o(8 * T), oo_c = take_o(16 * T), oo_t = take_o(4 * T),
               oo_s = take_o(48 * T);
  CU(c->d_ba_out.ensure(oo + 256));
  char *out = c->d_ba_out.as<char>();
  CU(cudaEventRecord(c->ev0, s));
  // per-track prologue on the device: minimal parameterisation of the start lines, constant-track flags
  lm::launch_zero_words(in + o_err, 8, s);
  lm::launch_lm_prologue(reinterpret_cast<const double *>(in + o_li), reinterpret_cast<const int64_t *>(in + o_so),
                         reinterpret_cast<const int32_t *>(in + o_sv), T, cfg->min_num_images,
                         reinterpret_cast<double *>(in + o_x), reinterpret_cast<uint8_t *>(in + o_a),
                         reinterpret_cast<int *>(in + o_err), s);
  lm::launch_lm_prepare(reinterpret_cast<const double *>(in + o_s), reinterpret_cast<const int32_t *>(in + o_sv),
                        reinterpret_cast<const double *>(in + o_k), reinterpret_cast<const double *>(in + o_q),
                        reinterpret_cast<const double *>(in + o_t),
                        (sup_vp && n) ? reinterpret_cast<const double *>(in + o_vp) : nullptr, cfg->vp_multiplier, n,
                        c->d_ba_blocks.as<lm::LMBlockDev>(), s);
  CU(cudaEventRecord(c->evk0, s));
  lm::LMParams p;
  p.blocks = c->d_ba_blocks.as<lm::LMBlockDev>();
  p.sup_off = reinterpret_cast<const int64_t *>(in + o_so);
  p.x0 = reinterpret_cast<const double *>(in + o_x);
  p.active = reinterpret_cast<const uint8_t *>(in + o_a);
  p.x_out = reinterpret_cast<double *>(out + oo_x);
  p.iters = reinterpret_cast<int32_t *>(out + oo_i);
  p.cost = reinterpret_cast<double *>(out + oo_c);
  p.term = reinterpret_cast<int32_t *>(out + oo_t);
  p.line3d = dev_seg ? reinterpret_cast<const double *>(in + o_l3) : nullptr;
  p.seg_out = dev_seg ? reinterpret_cast<double *>(out + oo_s) : nullptr;
  p.next_track = reinterpret_cast<unsigned long long *>(in + o_err + 16);
  p.num_outliers = cfg->num_outliers;
  p.T = T;
  p.geometric_alpha = cfg->geometric_alpha;
  p.cauchy_scale = cfg->cauchy_scale;
  p.max_num_iterations = cfg->max_num_iterations;
  p.max_invalid = cfg->max_num_consecutive_invalid_steps;
  lm::launch_lm_refine(p, s);
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->evk1, s));
  // results land in a pinned staging area of the context (a pageable destination would serialise the copies)
  const size_t T1 = (size_t)std::max<int64_t>(T, 1);
  const size_t need_pin = T1 * (48 + 16 + 8 + 48) + 64;
  if (need_pin > c->h_ba_pin_cap) {
    if (c->h_ba_pin) cudaFreeHost(c->h_ba_pin);
    c->h_ba_pin = nullptr;
    c->h_ba_pin_cap = 0;
    CU(cudaHostAlloc(&c->h_ba_pin, need_pin + need_pin / 4, cudaHostAllocDefault));
    c->h_ba_pin_cap = need_pin + need_pin / 4;
  }
  double *xf = reinterpret_cast<double *>(c->h_ba_pin);
  double *cost = xf + 6 * T1;
  double *segd = cost + 2 * T1;
  int32_t *iters = reinterpret_cast<int32_t *>(segd + 6 * T1);
  int *h_err = reinterpret_cast<int *>(iters + 2 * T1);
  *h_err = 0;
  if (T) {
    if (dev_seg) CU(cudaMemcpyAsync(segd, out + oo_s, 48 * T, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(xf, out + oo_x, 48 * T, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(iters, out + oo_i, 8 * T, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(cost, out + oo_c, 16 * T, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(h_err, in + o_err, 4, cudaMemcpyDeviceToHost, s));
  }
  CU(cudaStreamSynchronize(s));
  if (*h_err) return fail(LM_ERR_INVALID, "track with a zero-length 3D line (CHECK_GT(line.length(), 0))");
  float ms0 = 0, ms1 = 0;
  CU(cudaEventElapsedTime(&ms0, c->ev0, c->evk0));
  CU(cudaEventElapsedTime(&ms1, c->evk0, c->evk1));
  c->stats.n_kernel_launches += 4;
  c->ba_stats.n_tracks = T;
  c->ba_stats.n_blocks = n;
  c->ba_stats.prepare_ms = ms0;
  c->ba_stats.solve_ms = ms1;
  c->ba_stats.total_iterations = c->ba_stats.total_successful = 0;
  for (int64_t t = 0; t < T; ++t) {
    c->ba_stats.total_iterations += iters[2 * t];
    c->ba_stats.total_successful += iters[2 * t + 1];
    if (out_minimal) memcpy(out_minimal + 6 * t, &xf[6 * t], 48);
    if (out_iters) { out_iters[2 * t] = iters[2 * t]; out_iters[2 * t + 1] = iters[2 * t + 1]; }
    if (out_cost) { out_cost[2 * t] = cost[2 * t]; out_cost[2 * t + 1] = cost[2 * t + 1]; }
    if (out_line && dev_seg && !std::isnan(segd[6 * t])) {
      memcpy(out_line + 6 * t, &segd[6 * t], 48); // cut on the device
    } else if (out_line) {
      const int64_t a = sup_off[t], b = sup_off[t + 1];
      if (b > a && 2 * (b - a) - 1 - cfg->num_outliers >= 0 && cfg->num_outliers < 2 * (b - a))
        segment_from_minimal(&xf[6 * t], line3d + 6 * a, b - a, cfg->num_outliers, out_line + 6 * t);
      else
        memcpy(out_line + 6 * t, line_init + 6 * t, 48);
    }
  }
  return LM_OK;
}

int lm_ba_get_stats(lm_ctx *c, lm_ba_stats *out) {
  if (!c || !out) return fail(LM_ERR_INVALID, "NULL argument");
  *out = c->ba_stats;
  return LM_OK;
}

} // extern "C"

// ---- vanishing points ----------------------------------------------------------------------------
namespace {

struct L2h { double x1, y1, x2, y2; };
inline double len_h(const L2h &l) { return std::sqrt((l.x1 - l.x2) * (l.x1 - l.x2) + (l.y1 - l.y2) * (l.y1 - l.y2)); }
// Line2d::coords (base/linebase.cc:35-39)
inline void coords_h(const L2h &l, double c[3]) {
  c[0] = l.y1 - l.y2; c[1] = l.x2 - l.x1; c[2] = l.x1 * l.y2 - l.x2 * l.y1;
  const double n2 = c[0] * c[0] + c[1] * c[1] + c[2] * c[2];
  if (n2 > 0) { const double n = std::sqrt(n2); c[0] /= n; c[1] /= n; c[2] /= n; }
}
// BaseVPDetector::count_valid_supports_2d (vplib/base_vp_detector.cc:41-73)
int count_valid_supports_2d_h(const std::vector<L2h> &lines, double th_perp) {
  const size_t n = lines.size();
  std::vector<int> parent(n, -1);
  auto root = [&](size_t i) { while (parent[i] != -1) i = parent[i]; return i; };
  auto dist = [&](const L2h &l, double qx, double qy) {
    double c[3];
    coords_h(l, c);
    return std::fabs(c[0] * qx + c[1] * qy + c[2]) / std::sqrt(c[0] * c[0] + c[1] * c[1]);
  };
  for (size_t i = 0; i + 1 < n; ++i) {
    const size_t ri = root(i);
    for (size_t j = i + 1; j < n; ++j) {
      const size_t rj = root(j);
      if (rj == ri) continue;
      size_t k1 = i, k2 = j;
      if (len_h(lines[i]) > len_h(lines[j])) { k1 = j; k2 = i; }
      const double ds = dist(lines[k2], lines[k1].x1, lines[k1].y1), de = dist(lines[k2], lines[k1].x2, lines[k1].y2);
      if (((ds < de) ? de : ds) > th_perp) continue;
      parent[rj] = (int)ri;
    }
  }
  int cnt = 0;
  for (size_t i = 0; i < n; ++i) cnt += parent[i] == -1;
  return cnt;
}
// JLinkage::fitVP (JLinkage.cc:86-100): right singular vector of the smallest singular value
void smallest_eigvec(const double Ain[3][3], double out[3]) {
  double A[3][3], V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  memcpy(A, Ain, sizeof(A));
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = A[0][1] * A[0][1] + A[0][2] * A[0][2] + A[1][2] * A[1][2];
    double diag = A[0][0] * A[0][0] + A[1][1] * A[1][1] + A[2][2] * A[2][2];
    if (off == 0 || off <= 1e-32 * diag) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (A[p][q] == 0) continue;
        double theta = (A[q][q] - A[p][p]) / (2 * A[p][q]);
        double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1));
        double cs = 1 / std::sqrt(t * t + 1), sn = t * cs;
        for (int k = 0; k < 3; ++k) { double a = A[k][p], b = A[k][q]; A[k][p] = cs * a - sn * b; A[k][q] = sn * a + cs * b; }
        for (int k = 0; k < 3; ++k) { double a = A[p][k], b = A[q][k]; A[p][k] = cs * a - sn * b; A[q][k] = sn * a + cs * b; }
        for (int k = 0; k < 3; ++k) { double a = V[k][p], b = V[k][q]; V[k][p] = cs * a - sn * b; V[k][q] = sn * a + cs * b; }
      }
  }
  int best = 0;
  if (A[1][1] < A[best][best]) best = 1;
  if (A[2][2] < A[best][best]) best = 2;
  double n = std::sqrt(V[0][best] * V[0][best] + V[1][best] * V[1][best] + V[2][best] * V[2][best]);
  for (int k = 0; k < 3; ++k) out[k] = V[k][best] / n;
}

} // namespace

extern "C" {

int64_t lm_vp_detect(lm_ctx *c, int32_t n_images, const int64_t *line_off, const double *segs, const lm_vp_config *cfg,
                     int32_t *labels, int64_t *vp_off, double *vps, int64_t vp_cap) {
  return lm_vp_detect_indexed(c, n_images, line_off, segs, cfg, nullptr, labels, vp_off, vps, vp_cap);
}
int lm_vp_get_stats(lm_ctx *c, lm_vp_stats *out) {
  if (!c || !out) return fail(LM_ERR_INVALID, "NULL argument");
  *out = c->vp_stats;
  return LM_OK;
}
int64_t lm_vp_detect_indexed(lm_ctx *c, int32_t n_images, const int64_t *line_off, const double *segs,
                             const lm_vp_config *cfg, const int64_t *image_index, int32_t *labels, int64_t *vp_off,
                             double *vps, int64_t vp_cap) {
  if (!c || !cfg || !line_off || !labels || !vp_off) return fail(LM_ERR_INVALID, "NULL argument");
  if (n_images < 0) return fail(LM_ERR_INVALID, "bad sizes");
  if (cfg->n_models <= 0 || cfg->n_models > 65535) return fail(LM_ERR_INVALID, "n_models must be in [1, 65535]");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  // ComputeVPLabels :17-36: segments of at least min_length px, cast to float
  std::vector<float> pts;
  std::vector<int64_t> valid_off(n_images + 1, 0);
  std::vector<int32_t> valid_ids;
  int max_n = 0;
  for (int im = 0; im < n_images; ++im) {
    for (int64_t l = line_off[im]; l < line_off[im + 1]; ++l) {
      const double *g = segs + 4 * l;
      const double len = std::sqrt((g[0] - g[2]) * (g[0] - g[2]) + (g[1] - g[3]) * (g[1] - g[3]));
      if (len < cfg->min_length) continue;
      valid_ids.push_back((int32_t)(l - line_off[im]));
      for (int k = 0; k < 4; ++k) pts.push_back((float)g[k]);
    }
    valid_off[im + 1] = (int64_t)valid_ids.size();
    max_n = std::max(max_n, (int)(valid_off[im + 1] - valid_off[im]));
  }
  if (max_n > 8192) return fail(LM_ERR_INVALID, "more than 8192 segments of min_length in one image");
  const int64_t nv = (int64_t)valid_ids.size();
  std::vector<int32_t> raw(std::max<int64_t>(nv, 1), -1), ncl(std::max(n_images, 1), 0);
  const int min_lines = 2 * std::max(cfg->min_num_supports, 10);
  bool vp_kernel_ran = false;
  if (nv > 0 && max_n >= min_lines) {
    const int W = (cfg->n_models + 31) / 32;
    int grid = std::min(n_images, c->sm_count * 2);
    CU(c->d_vp_pts.ensure(16 * nv));
    CU(c->d_vp_off.ensure(8 * (n_images + 1)));
    CU(c->d_vp_labels.ensure(4 * nv));
    CU(c->d_vp_nc.ensure(4 * n_images));
    CU(c->d_vp_ps.ensure((size_t)grid * max_n * W * 4));
    CU(c->d_vp_mat.ensure((size_t)grid * max_n * max_n * 4));
    CU(c->d_vp_idx.ensure(8 * std::max(n_images, 1)));
    CU(cudaMemcpyAsync(c->d_vp_pts.p, pts.data(), 16 * nv, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(c->d_vp_off.p, valid_off.data(), 8 * (n_images + 1), cudaMemcpyHostToDevice, s));
    if (image_index) CU(cudaMemcpyAsync(c->d_vp_idx.p, image_index, 8 * n_images, cudaMemcpyHostToDevice, s));
    lm::VPParams p;
    p.pts = c->d_vp_pts.as<float4>();
    p.valid_off = c->d_vp_off.as<int64_t>();
    p.image_index = image_index ? c->d_vp_idx.as<int64_t>() : nullptr;
    p.labels = c->d_vp_labels.as<int32_t>();
    p.n_clusters = c->d_vp_nc.as<int32_t>();
    p.ps_slab = c->d_vp_ps.as<uint32_t>();
    p.mat_slab = c->d_vp_mat.as<uint32_t>();
    p.n_images = n_images; p.n_models = cfg->n_models; p.max_n = max_n; p.min_lines = min_lines;
    p.inlier_threshold = (float)cfg->inlier_threshold;
    p.seed = cfg->seed;
    if (lm::vp_smem_bytes(p.n_models, p.max_n) > (size_t)c->max_smem_optin)
      return fail(LM_ERR_INVALID, "n_models too large for shared memory");
    CU(cudaEventRecord(c->evk0, s));
    lm::launch_jlinkage(p, grid, s);
    CU(cudaEventRecord(c->evk1, s));
    CU(cudaGetLastError());
    vp_kernel_ran = true;
    c->stats.n_kernel_launches += 1;
    CU(cudaMemcpyAsync(raw.data(), c->d_vp_labels.p, 4 * nv, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(ncl.data(), c->d_vp_nc.p, 4 * n_images, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
  }
  // JLinkage.cc:56-83 (cluster filtering) and AssociateVPs :102-127 (VP fitting), per image on the host
  int64_t n_vps = 0;
  for (int im = 0; im < n_images; ++im) {
    vp_off[im] = n_vps;
    const int64_t L = line_off[im + 1] - line_off[im];
    int32_t *lab = labels + line_off[im];
    for (int64_t l = 0; l < L; ++l) lab[l] = -1;
    const int64_t v0 = valid_off[im], v1 = valid_off[im + 1];
    const int nc = ncl[im];
    if (nc <= 0 || v1 - v0 < min_lines) continue;
    std::vector<std::vector<L2h>> sup(nc);
    for (int64_t k = v0; k < v1; ++k) {
      if (raw[k] < 0) continue;
      const double *g = segs + 4 * (line_off[im] + valid_ids[k]);
      sup[raw[k]].push_back(L2h{g[0], g[1], g[2], g[3]});
    }
    std::vector<int> vp_ids(nc, -1);
    int counter = 0;
    for (int q = 0; q < nc; ++q) {
      if ((int)sup[q].size() < cfg->min_num_supports) continue;
      if (count_valid_supports_2d_h(sup[q], cfg->th_perp_supports) < cfg->min_num_supports) continue;
      vp_ids[q] = counter++;
    }
    std::vector<std::array<double, 9>> S(counter, std::array<double, 9>{});
    for (int64_t k = v0; k < v1; ++k) {
      if (raw[k] < 0 || vp_ids[raw[k]] < 0) continue;
      const int v = vp_ids[raw[k]];
      lab[valid_ids[k]] = v;
      const double *g = segs + 4 * (line_off[im] + valid_ids[k]);
      double cc[3];
      coords_h(L2h{g[0], g[1], g[2], g[3]}, cc);
      for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) S[v][3 * a + b] += cc[a] * cc[b];
    }
    for (int v = 0; v < counter; ++v) {
      double A[3][3], e[3];
      for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) A[a][b] = S[v][3 * a + b];
      smallest_eigvec(A, e);
      if (vps && n_vps < vp_cap) { vps[3 * n_vps] = e[0]; vps[3 * n_vps + 1] = e[1]; vps[3 * n_vps + 2] = e[2]; }
      ++n_vps;
    }
  }
  vp_off[n_images] = n_vps;
  c->vp_stats.n_images = n_images;
  c->vp_stats.n_segments = nv;
  c->vp_stats.n_vps = n_vps;
  c->vp_stats.kernel_ms = 0;
  if (vp_kernel_ran) { float ms = 0; CU(cudaEventElapsedTime(&ms, c->evk0, c->evk1)); c->vp_stats.kernel_ms = ms; }
  return n_vps;
}

// ---- track filters + remerge (merging/merging_utils.cc, merging/merging.cc:513-645) -------------------
int lm_tracks_support_flags(lm_ctx *c, int32_t n_views, const int32_t *model_ids, const double *kvec, const double *qvec,
                            const double *tvec, int64_t T, const int64_t *sup_off, const int32_t *sup_view,
                            const double *segs, const double *track_line, const lm_filter_config *cfg,
                            uint8_t *out_flags) {
  if (!c || !cfg || !sup_off || !kvec || !qvec || !tvec) return fail(LM_ERR_INVALID, "NULL argument");
  if (T < 0 || n_views <= 0) return fail(LM_ERR_INVALID, "bad sizes");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const int64_t n = sup_off[T];
  if (n == 0) return LM_OK;
  if (!sup_view || !segs || !track_line || !out_flags) return fail(LM_ERR_INVALID, "NULL argument");
  for (int64_t k = 0; k < n; ++k)
    if (sup_view[k] < 0 || sup_view[k] >= n_views) return fail(LM_ERR_INVALID, "support view index out of range");
  std::vector<lm::ViewD> views(n_views);
  for (int v = 0; v < n_views; ++v) {
    const int mid = model_ids ? model_ids[v] : 1;
    if (mid != 0 && mid != 1) return fail(LM_ERR_INVALID, "only SIMPLE_PINHOLE / PINHOLE are legal on this path");
    make_view(mid, kvec + 4 * v, qvec + 4 * v, tvec + 3 * v, views[v]);
  }
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const size_t o_v = take(sizeof(lm::ViewD) * n_views), o_s = take(32 * n), o_so = take(8 * (T + 1)), o_sv = take(4 * n),
               o_tl = take(48 * T);
  CU(c->d_mg_in.ensure(off + 256));
  CU(c->d_mg_out.ensure(n + 256));
  char *in = c->d_mg_in.as<char>();
  CU(cudaEventRecord(c->ev0, s));
  CU(cudaMemcpyAsync(in + o_v, views.data(), sizeof(lm::ViewD) * n_views, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_s, segs, 32 * n, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_so, sup_off, 8 * (T + 1), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_sv, sup_view, 4 * n, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_tl, track_line, 48 * T, cudaMemcpyHostToDevice, s));
  lm::SupportParams p;
  p.views = reinterpret_cast<const lm::ViewD *>(in + o_v);
  p.sup_off = reinterpret_cast<const int64_t *>(in + o_so);
  p.sup_view = reinterpret_cast<const int32_t *>(in + o_sv);
  p.segs = reinterpret_cast<const double4 *>(in + o_s);
  p.track_line = reinterpret_cast<const double *>(in + o_tl);
  p.T = T; p.S = n;
  p.th_angular2d = cfg->th_angular_2d; p.th_perp2d = cfg->th_perp_2d;
  p.th_sv_angular3d = cfg->th_sv_angular_3d; p.th_overlap = cfg->th_overlap;
  p.flags = c->d_mg_out.as<uint8_t>();
  CU(cudaEventRecord(c->evk0, s));
  lm::launch_support_flags(p, s);
  CU(cudaEventRecord(c->evk1, s));
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out_flags, p.flags, n, cudaMemcpyDeviceToHost, s));
  CU(cudaEventRecord(c->ev1, s));
  CU(cudaStreamSynchronize(s));
  float ms = 0, msk = 0;
  CU(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  CU(cudaEventElapsedTime(&msk, c->evk0, c->evk1));
  c->mg_stats.n_supports = n;
  c->mg_stats.last_flags_ms = ms;
  c->mg_stats.last_flags_kernel_ms = msk;
  c->mg_stats.n_kernel_launches += 1;
  return LM_OK;
}

int lm_aggregate_lines(int64_t T, const int64_t *off, const double *lines, const double *scores, int32_t num_outliers,
                       double *out_line) {
  if (T < 0 || !off || !out_line) return fail(LM_ERR_INVALID, "NULL argument");
  if (num_outliers < 0) return fail(LM_ERR_INVALID, "num_outliers must be >= 0");
  std::vector<AggItem> it;
  for (int64_t t = 0; t < T; ++t) {
    const int64_t n = off[t + 1] - off[t];
    double *o = out_line + 7 * t;
    if (n <= 0) { memset(o, 0, 7 * sizeof(double)); continue; }
    if (n >= 4 && 2 * n - 1 - num_outliers < num_outliers) return fail(LM_ERR_INVALID, "num_outliers too large for a group");
    it.resize(n);
    for (int64_t k = 0; k < n; ++k) it[k] = AggItem{lines + 7 * (off[t] + k), lines[7 * (off[t] + k) + 6], scores[off[t] + k]};
    aggregate_items(it, num_outliers, o);
  }
  return LM_OK;
}

int64_t lm_remerge_labels(lm_ctx *c, int64_t T, const double *track_line, const uint8_t *active,
                          const lm_linker_config *linker3d, int32_t *out_labels, int64_t *out_n_edges) {
  if (!c || !linker3d) return fail(LM_ERR_INVALID, "NULL argument");
  if (T < 0 || T >= ((int64_t)1 << 31)) return fail(LM_ERR_INVALID, "bad track count");
  if (out_n_edges) *out_n_edges = 0;
  if (T == 0) return 0;
  if (!track_line || !active || !out_labels) return fail(LM_ERR_INVALID, "NULL argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  lm_linker_config l3 = *linker3d; // set_to_spatial_merging (line_linker.h:123-129)
  l3.use_angle = 1; l3.use_overlap = 1; l3.use_perp = 0; l3.use_innerseg = 1; l3.use_scaleinv = 0;
  int64_t n_active = 0;
  for (int64_t t = 0; t < T; ++t) n_active += active[t] ? 1 : 0;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const size_t o_l = take(56 * T), o_d = take(16 * T), o_b = take(16 * T), o_a = take(T), o_c = take(16);
  CU(c->d_mg_in.ensure(off + 256));
  char *in = c->d_mg_in.as<char>();
  CU(cudaEventRecord(c->ev0, s));
  CU(cudaMemcpyAsync(in + o_l, track_line, 56 * T, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_a, active, T, cudaMemcpyHostToDevice, s));
  lm::RemergeParams p;
  p.lines = reinterpret_cast<const double *>(in + o_l);
  p.dirf = reinterpret_cast<const float4 *>(in + o_d);
  p.ballf = reinterpret_cast<const float4 *>(in + o_b);
  p.active = reinterpret_cast<const uint8_t *>(in + o_a);
  p.T = T;
  p.all_active = (n_active == T) ? 1 : 0;
  p.lk = to_dev<double>(l3);
  p.use_gate = (l3.th_angle > 0.0 && l3.th_angle < 89.0) ? 1 : 0;
  p.cos_gate = p.use_gate ? (float)(std::cos(l3.th_angle * 3.14159265358979323846 / 180.0) - 1e-5) : -1.0f;
  p.counter = reinterpret_cast<unsigned long long *>(in + o_c);
  p.use_ball = (l3.use_innerseg && l3.th_innerseg >= 0.0 && l3.score_th > 0.0 && l3.score_th < 1.0) ? 1 : 0;
  double origin[3] = {0, 0, 0}; // mean midpoint: keeps the fp32 coordinates of the ball gate small
  {
    int64_t nfin = 0;
    for (int64_t t = 0; t < T; ++t) {
      const double *l = track_line + 7 * t;
      const double m[3] = {0.5 * (l[0] + l[3]), 0.5 * (l[1] + l[4]), 0.5 * (l[2] + l[5])};
      if (std::isfinite(m[0]) && std::isfinite(m[1]) && std::isfinite(m[2])) { origin[0] += m[0]; origin[1] += m[1]; origin[2] += m[2]; ++nfin; }
    }
    if (nfin) for (int k = 0; k < 3; ++k) origin[k] /= (double)nfin;
  }
  lm::launch_remerge_dirs(p.lines, T, origin, l3.th_innerseg, reinterpret_cast<float4 *>(in + o_d),
                          reinterpret_cast<float4 *>(in + o_b), s);
  unsigned long long cap = (unsigned long long)std::max<int64_t>(4 * T, 1 << 16);
  unsigned long long cnt[2] = {0, 0};
  float msk = 0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    CU(c->d_mg_edges.ensure(8 * cap));
    p.edges = c->d_mg_edges.as<uint32_t>();
    p.capacity = cap;
    lm::launch_zero_words(reinterpret_cast<unsigned int *>(in + o_c), 4, s);
    CU(cudaEventRecord(c->evk0, s));
    if (n_active > 0) lm::launch_remerge_pairs(p, s);
    CU(cudaEventRecord(c->evk1, s));
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(cnt, p.counter, 16, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    CU(cudaEventElapsedTime(&msk, c->evk0, c->evk1));
    c->mg_stats.n_kernel_launches += 3;
    if (cnt[0] <= cap) break;
    cap = cnt[0]; // the list overflowed: run again with the exact size
  }
  const int64_t ne = (int64_t)cnt[0];
  std::vector<uint32_t> h_edges(2 * std::max<int64_t>(ne, 1));
  if (ne) CU(cudaMemcpyAsync(h_edges.data(), p.edges, 8 * ne, cudaMemcpyDeviceToHost, s));
  CU(cudaEventRecord(c->ev1, s));
  CU(cudaStreamSynchronize(s));
  float ms = 0;
  CU(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  // std::set<pair> iteration order = lexicographic (merging.cc:558-560)
  std::vector<uint64_t> keys(ne);
  for (int64_t e = 0; e < ne; ++e) keys[e] = ((uint64_t)h_edges[2 * e] << 32) | h_edges[2 * e + 1];
  std::sort(keys.begin(), keys.end());
  // union-find with the group-size heuristic (merging.cc:562-589)
  std::vector<int> parent(T, -1);
  std::vector<int64_t> gsize(T, 1);
  for (int64_t e = 0; e < ne; ++e) {
    const size_t r1 = uf_root((size_t)(keys[e] >> 32), parent), r2 = uf_root((size_t)(keys[e] & 0xffffffffu), parent);
    if (r1 == r2) continue;
    if (gsize[r1] < gsize[r2]) { parent[r1] = (int)r2; gsize[r2] += gsize[r1]; gsize[r1] = 0; }
    else { parent[r2] = (int)r1; gsize[r1] += gsize[r2]; gsize[r2] = 0; }
  }
  int64_t n_groups = 0;
  for (int64_t t = 0; t < T; ++t) out_labels[t] = (parent[t] == -1) ? (int32_t)(n_groups++) : -1;
  for (int64_t t = 0; t < T; ++t)
    if (out_labels[t] == -1) out_labels[t] = out_labels[uf_root((size_t)t, parent)];
  if (out_n_edges) *out_n_edges = ne;
  c->mg_stats.n_tracks = T;
  c->mg_stats.n_pairs_gated = (int64_t)cnt[1];
  c->mg_stats.n_edges = ne;
  c->mg_stats.last_remerge_ms = ms;
  c->mg_stats.last_remerge_kernel_ms = msk;
  return n_groups;
}

int lm_merge_get_stats(lm_ctx *c, lm_merge_stats *out) {
  if (!c || !out) return fail(LM_ERR_INVALID, "NULL argument");
  *out = c->mg_stats;
  return LM_OK;
}

} // extern "C"

// ---- visual-neighbour ranking and robust ranges from a sparse point model (SURVEY.md 8 f4) -------------------------
extern "C" {

int lm_sfm_rank_neighbors(lm_ctx *c, int32_t n_images, const double *centres, int64_t n_points, const double *xyz,
                          const int64_t *track_off, const int32_t *track_img, int32_t num_images,
                          double min_triangulation_angle_deg, int32_t mode, int32_t *out_neighbors, int32_t *out_count) {
  if (!c || !centres || !track_off || !out_neighbors || !out_count) return fail(LM_ERR_INVALID, "NULL argument");
  if (n_images <= 0 || n_images > 65535 || n_points < 0 || num_images <= 0 || mode < 0 || mode > 2)
    return fail(LM_ERR_INVALID, "bad sizes");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const int64_t n_ent = track_off[n_points];
  for (int64_t e = 0; e < n_ent; ++e)
    if (track_img[e] < 0 || track_img[e] >= n_images) return fail(LM_ERR_INVALID, "track image index out of range");
  // records per point: pairs of its track entries
  std::vector<int64_t> rec_off(n_points + 1, 0);
  for (int64_t p = 0; p < n_points; ++p) {
    const int64_t t = track_off[p + 1] - track_off[p];
    rec_off[p + 1] = rec_off[p] + t * (t - 1) / 2;
  }
  const int64_t n_rec = rec_off[n_points];
  if (n_rec >= ((int64_t)1 << 31) - 64) return fail(LM_ERR_INVALID, "more than 2^31 (point, image pair) records");
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const size_t o_c = take(24 * (size_t)n_images), o_x = take(24 * (size_t)std::max<int64_t>(n_points, 1)),
               o_to = take(8 * (size_t)(n_points + 1)), o_ti = take(4 * (size_t)std::max<int64_t>(n_ent, 1)),
               o_ro = take(8 * (size_t)(n_points + 1)), o_np = take(4 * (size_t)n_images), o_sc = take(64),
               o_out = take(4 * (size_t)n_images * num_images), o_cnt = take(4 * (size_t)n_images);
  CU(c->d_sfm_in.ensure(off + 256));
  char *in = c->d_sfm_in.as<char>();
  CU(cudaMemcpyAsync(in + o_c, centres, 24 * (size_t)n_images, cudaMemcpyHostToDevice, s));
  if (n_points) CU(cudaMemcpyAsync(in + o_x, xyz, 24 * (size_t)n_points, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_to, track_off, 8 * (size_t)(n_points + 1), cudaMemcpyHostToDevice, s));
  if (n_ent) CU(cudaMemcpyAsync(in + o_ti, track_img, 4 * (size_t)n_ent, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(in + o_ro, rec_off.data(), 8 * (size_t)(n_points + 1), cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(in + o_np, 0, 4 * (size_t)n_images, s));
  CU(cudaMemsetAsync(in + o_sc, 0, 64, s));
  unsigned int *d_np = reinterpret_cast<unsigned int *>(in + o_np);
  unsigned int *d_ndir = reinterpret_cast<unsigned int *>(in + o_sc);
  int *d_nruns = reinterpret_cast<int *>(in + o_sc + 16);
  int64_t n_dir = 0;
  if (n_rec > 0) {
    // (a pair seen once yields two directed records: the scratch is sized for 2 n_rec)
    CU(c->d_sfm_keys.ensure(16 * (size_t)n_rec));
    CU(c->d_sfm_keys2.ensure(16 * (size_t)n_rec));
    lm::launch_sfm_pair_keys(reinterpret_cast<const double *>(in + o_c), reinterpret_cast<const double *>(in + o_x),
                             reinterpret_cast<const int64_t *>(in + o_to), reinterpret_cast<const int32_t *>(in + o_ti),
                             reinterpret_cast<const int64_t *>(in + o_ro), n_points, n_rec,
                             c->d_sfm_keys.as<unsigned long long>(), d_np, s);
    cub::DoubleBuffer<unsigned long long> dk(c->d_sfm_keys.as<unsigned long long>(), c->d_sfm_keys2.as<unsigned long long>());
    size_t tmp = 0;
    CU(cub::DeviceRadixSort::SortKeys(nullptr, tmp, dk, (int)n_rec, 0, 64, s));
    CU(c->d_sort_tmp.ensure(tmp));
    CU(cub::DeviceRadixSort::SortKeys(c->d_sort_tmp.p, tmp, dk, (int)n_rec, 0, 64, s));
    const unsigned long long *sorted = dk.Current();
    // runs of equal image pairs: ids -> run-length encode -> starts
    CU(c->d_sfm_a.ensure(8 * (size_t)n_rec));       // pair ids, later the directed records
    CU(c->d_sfm_b.ensure(8 * (size_t)n_rec + 16));  // unique pairs, later the sort's alternate buffer
    CU(c->d_sfm_c.ensure(4 * (size_t)n_rec + 16));  // run lengths
    CU(c->d_sfm_d.ensure(4 * (size_t)n_rec + 16));  // run starts
    lm::launch_sfm_pair_ids(sorted, n_rec, c->d_sfm_a.as<unsigned int>(), s);
    size_t tmp2 = 0;
    CU(cub::DeviceRunLengthEncode::Encode(nullptr, tmp2, c->d_sfm_a.as<unsigned int>(), c->d_sfm_b.as<unsigned int>(),
                                          c->d_sfm_c.as<unsigned int>(), d_nruns, (int)n_rec, s));
    CU(c->d_sort_tmp.ensure(tmp2));
    CU(cub::DeviceRunLengthEncode::Encode(c->d_sort_tmp.p, tmp2, c->d_sfm_a.as<unsigned int>(), c->d_sfm_b.as<unsigned int>(),
                                          c->d_sfm_c.as<unsigned int>(), d_nruns, (int)n_rec, s));
    int n_runs = 0;
    CU(cudaMemcpyAsync(&n_runs, d_nruns, 4, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    size_t tmp3 = 0;
    CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp3, c->d_sfm_c.as<unsigned int>(), c->d_sfm_d.as<unsigned int>(), n_runs, s));
    CU(c->d_sort_tmp.ensure(tmp3));
    CU(cub::DeviceScan::ExclusiveSum(c->d_sort_tmp.p, tmp3, c->d_sfm_c.as<unsigned int>(), c->d_sfm_d.as<unsigned int>(), n_runs, s));
    // directed (source, destination) records of the pairs that pass the angle test; the sorted keys are dead afterwards,
    // so their buffers carry the records: values in d_sfm_a (reused), keys in the alternate key buffer
    unsigned int *dir_val = c->d_sfm_a.as<unsigned int>();
    unsigned long long *dir_key = dk.Alternate();
    const float min_angle = (float)(min_triangulation_angle_deg * 3.14159265358979323846 / 180.0);
    lm::launch_sfm_scores(sorted, c->d_sfm_b.as<unsigned int>(), c->d_sfm_c.as<unsigned int>(), c->d_sfm_d.as<unsigned int>(),
                          n_runs, d_np, min_angle, mode, dir_val, dir_key, d_ndir, s);
    unsigned int h_ndir = 0;
    CU(cudaMemcpyAsync(&h_ndir, d_ndir, 4, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    n_dir = h_ndir;
    if (n_dir > 0) {
      // order: source ascending, score descending, destination ascending = three stable radix sorts, least significant first
      unsigned int *val2 = c->d_sfm_b.as<unsigned int>();
      unsigned long long *key2 = const_cast<unsigned long long *>(sorted); // the sorted pair keys are dead now
      {
        cub::DoubleBuffer<unsigned int> k(dir_val, val2);
        cub::DoubleBuffer<unsigned long long> v(dir_key, key2);
        size_t t1 = 0;
        CU(cub::DeviceRadixSort::SortPairs(nullptr, t1, k, v, (int)n_dir, 0, 32, s)); // by (source, destination)
        CU(c->d_sort_tmp.ensure(t1));
        CU(cub::DeviceRadixSort::SortPairs(c->d_sort_tmp.p, t1, k, v, (int)n_dir, 0, 32, s));
        cub::DoubleBuffer<unsigned long long> k2(v.Current(), v.Alternate());
        cub::DoubleBuffer<unsigned int> v2(k.Current(), k.Alternate());
        size_t t2 = 0;
        CU(cub::DeviceRadixSort::SortPairs(nullptr, t2, k2, v2, (int)n_dir, 0, 64, s)); // by score, descending
        CU(c->d_sort_tmp.ensure(t2));
        CU(cub::DeviceRadixSort::SortPairs(c->d_sort_tmp.p, t2, k2, v2, (int)n_dir, 0, 64, s));
        cub::DoubleBuffer<unsigned int> k3(v2.Current(), v2.Alternate());
        size_t t3 = 0;
        CU(cub::DeviceRadixSort::SortKeys(nullptr, t3, k3, (int)n_dir, 16, 32, s)); // by source (stable)
        CU(c->d_sort_tmp.ensure(t3));
        CU(cub::DeviceRadixSort::SortKeys(c->d_sort_tmp.p, t3, k3, (int)n_dir, 16, 32, s));
        dir_val = k3.Current();
      }
    }
    lm::launch_sfm_take(dir_val, n_dir, n_images, num_images, reinterpret_cast<int32_t *>(in + o_out),
                        reinterpret_cast<int32_t *>(in + o_cnt), s);
  } else {
    lm::launch_sfm_take(nullptr, 0, n_images, num_images, reinterpret_cast<int32_t *>(in + o_out),
                        reinterpret_cast<int32_t *>(in + o_cnt), s);
  }
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out_neighbors, in + o_out, 4 * (size_t)n_images * num_images, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(out_count, in + o_cnt, 4 * (size_t)n_images, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  c->stats.n_kernel_launches += 12;
  return LM_OK;
}

int lm_sfm_robust_ranges(lm_ctx *c, int64_t n_points, const double *xyz, double q_lo, double q_hi, double kstretch,
                         double out[6]) {
  if (!c || !xyz || !out) return fail(LM_ERR_INVALID, "NULL argument");
  if (n_points <= 0 || n_points >= ((int64_t)1 << 31) - 64) return fail(LM_ERR_INVALID, "bad point count");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  // SfmModel::ComputeRanges keeps the coordinates as float (sfm_model.cc:245-252): one float column per axis, sorted
  std::vector<float> col((size_t)n_points);
  CU(c->d_sfm_a.ensure(4 * (size_t)n_points));
  CU(c->d_sfm_b.ensure(4 * (size_t)n_points));
  for (int ax = 0; ax < 3; ++ax) {
    for (int64_t p = 0; p < n_points; ++p) col[p] = (float)xyz[3 * p + ax];
    CU(cudaMemcpyAsync(c->d_sfm_a.p, col.data(), 4 * (size_t)n_points, cudaMemcpyHostToDevice, s));
    cub::DoubleBuffer<float> dk(c->d_sfm_a.as<float>(), c->d_sfm_b.as<float>());
    size_t tmp = 0;
    CU(cub::DeviceRadixSort::SortKeys(nullptr, tmp, dk, (int)n_points, 0, 32, s));
    CU(c->d_sort_tmp.ensure(tmp));
    CU(cub::DeviceRadixSort::SortKeys(c->d_sort_tmp.p, tmp, dk, (int)n_points, 0, 32, s));
    const float kmin = (float)q_lo, kmax = (float)q_hi;
    const size_t i_lo = (size_t)((float)n_points * kmin), i_hi = (size_t)((float)n_points * kmax); // data[data.size() * k]
    float lo = 0, hi = 0;
    CU(cudaMemcpyAsync(&lo, dk.Current() + std::min<size_t>(i_lo, n_points - 1), 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(&hi, dk.Current() + std::min<size_t>(i_hi, n_points - 1), 4, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    const float ks = (float)kstretch, diff = hi - lo;
    lo -= ks * diff;
    hi += ks * diff;
    out[ax] = lo;
    out[3 + ax] = hi;
  }
  c->stats.n_kernel_launches += 12;
  return LM_OK;
}

} // extern "C"
