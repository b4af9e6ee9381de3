// tri_kernels.cuh — device-side data layout and kernel declarations of the triangulation path.
#pragma once
#include "lm_math.cuh"

namespace lm {

// Per-view constants, precomputed once in fp64 at lm_scene_upload and resident in HBM
// (replaces the per-call CameraView::R()/K_inv() recomputation of base/camera.h:72-73,106-110).
//   M = R^T K^-1   (ray(p) = normalize(M [p;1]), base/camera_view.cc:67-69)
//   C = -R^T T     (base/camera.h:109)
//   P = K [R|T]    (projection, base/camera_view.cc:61-65; row 2 = [R row 2 | T.z] gives projdepth)
//   fbar = f or (fx+fy)/2 (base/camera.cc:228-242; uncertainty = var2d * depth / fbar)
template <typename T> struct ViewT {
  T M[9];
  T C[3];
  T P[12];
  T fbar;
  T pad;
};
typedef ViewT<double> ViewD;
typedef ViewT<float> ViewF;

struct NodeRecord { // == lm_node_record
  double line[9];   // start3, end3, depths2, uncertainty
  double score;
  int32_t ng_view, ng_line, n_cand, n_valid;
};

// Kernel parameters of the fused generate+score+select kernel.
struct TriParams {
  const ViewD *views;          // [V]
  const double4 *segs;         // [sum L] x1,y1,x2,y2 (after add_halfpix)
  const uint16_t *node_view;   // [sum L] view index of each node
  const int64_t *line_off;     // [V+1] node offset of each view
  const uint32_t *row_ng;      // [rows] sorted by node: (ng_view << 16) | ng_line
  const uint32_t *node_row_off; // [nodes+1] row range of each node in row_ng
  const int32_t *vp_label;     // [sum L] VP label per line or NULL
  const int64_t *vp_off;       // [V+1]
  const double *vps;           // [sum n_vp][3]
  NodeRecord *nodes;           // [nodes] out
  uint8_t *row_state;          // [rows][ns] out: 0 rejected, 1 candidate, 2 valid connection (ns = 3 with VPs)
  double *row_cand;            // [rows][ns][10] out (debug_mode only, else NULL)
  unsigned long long *counters; // [4] n_candidates, n_valid, pairs past the 3d gates, pairs scored exactly
  int *overflow;               // set when a node has more candidate slots than `cap` (the host re-runs with the exact size)
  char *slab;                  // global scratch for nodes whose rows exceed the smem capacity (or NULL)
  int64_t slab_stride;         // bytes per CTA
  int64_t node_begin, node_end;
  int cap;                     // candidate capacity of the staging area
  int use_slab;
  // split path (tri_gen_kernel + tri_score_kernel) of one pipeline group
  const uint32_t *row_node;    // [rows] node of every row (the node-sorted keys)
  double *cand;                // candidate records of the group's slots, field-major (see tri_kernels.cu)
  int64_t cand_stride;         // slots per field
  int64_t row_begin, row_end;  // rows of the group
  unsigned int *max_cand;      // largest candidate count of a node in the run
  // config (triangulation/base_line_triangulator.h:22-43, global_line_triangulator.h:11-25)
  double min_length_2d, line_tri_angle_threshold, IoU_threshold, sensitivity_threshold, var2d, fullscore_th;
  int max_valid_conns, use_endpoints_triangulation, disable_algebraic, use_vp, disable_vp;
  int ranges_flag;
  double rlo[3], rhi[3];
  LinkerDev<double> l2d;  // user linker2d_config
  LinkerDev<double> l3d;  // linker3d_config after set_to_shared_parent_scoring()
  // pruning-gate constants derived from the thresholds (see tri_kernels.cu "pruning gates")
  float cos_th3d_f;       // cos(l3d.th_angle) - 4e-6
  double cos2_th2d;       // cos^2(l2d.th_angle) (0 when th_angle >= 90)
  double th_perp2_2d;     // l2d.th_perp^2
  double sin2_tri;        // sin^2(line_tri_angle_threshold); valid when tri_poly_ok
  double sin2_sens;       // sin^2(sensitivity_threshold); valid when sens_poly_ok
  int tri_poly_ok, sens_poly_ok; // thresholds inside (0, 90): the polynomial forms are equivalent
  // reduced-form scorer constants: 1/sigma of the angle / scale-invariance / perpendicular tests and the
  // largest q = (v/sigma)^2 that can still reach score_th (with a 1e-9 margin)
  int fast_forms;
  double inv_sig_a3, inv_sig_s3, inv_sig_a2, inv_sig_p2, q_cut3;
  double q_cut3_lo, q_cut2, q_cut2_lo; // -2 ln(score_th) * (1 -/+ 1e-9) of the two linkers
  double inv_smart_den2;               // 1 / (l2d.th_smartoverlap - l2d.th_overlap)
};

struct EdgeParams {
  const NodeRecord *nodes;
  const int64_t *edges; // [n][2] (a<b) node ids
  double *weight;       // [n] out
  int64_t n;
  LinkerDev<double> l3d; // linker3d_config after set_to_spatial_merging()
};

size_t tri_smem_bytes(int cap, bool fast);
void launch_group_edges(const uint8_t *row_state, const uint32_t *row_ng, const uint32_t *node_row_off,
                        const uint32_t *local_off, unsigned int *totals, int g, int64_t shard_node_begin, int64_t node_lo,
                        int64_t n, int ns, uint32_t *edge_off, uint32_t *edge_ng, cudaStream_t s);
void launch_scene_prepare(const double *segs_raw, int64_t n_nodes, double add, const int64_t *line_off, int n_views,
                          double *segs, uint16_t *node_view, cudaStream_t s);
cudaError_t launch_tri_node_kernel(const TriParams &p, int grid, int block, size_t smem, cudaStream_t s);
// Split form of the fast path: candidates of all rows of the group, then per-node scoring (p.cap sized from candidates).
static constexpr int kCandFields = 11; // fp64 fields of a candidate record
size_t tri_score_smem_bytes(int cap);
cudaError_t launch_tri_split(const TriParams &p, int grid, size_t smem, cudaStream_t s);
void launch_expand_rows(const int32_t *d_pairs, const int64_t *d_blk_row_off, const int32_t *d_blk_src_view,
                        const int32_t *d_blk_ng_view, const int64_t *d_blk_pair_off, int n_blocks,
                        const int64_t *d_line_off, int64_t r_begin, int64_t r_end, uint32_t *d_key, uint32_t *d_val,
                        int *d_err, cudaStream_t s);
void launch_expand_exhaustive(const int64_t *d_blk_row_off, const int32_t *d_blk_src_view,
                              const int32_t *d_blk_ng_view, int n_blocks, const int64_t *d_line_off,
                              int64_t n_rows, uint32_t *d_key, uint32_t *d_val, cudaStream_t s);
void launch_node_offsets(const uint32_t *d_sorted_key, int64_t n_rows, int64_t row_base, int64_t node_lo,
                         int64_t node_hi, uint32_t *d_node_row_off, unsigned int *d_max_rows, cudaStream_t s);
// Node-major rows by a per-view stable counting sort (non-exhaustive matches). A view with more lines than
// kRowSortMaxLines keeps the radix-sort path; kRowSortTile rows of a view form one tile (one CTA).
static constexpr int kRowSortMaxLines = 4096;
static constexpr int kRowSortTile = 8192;
size_t row_scatter_smem_bytes(int max_lines);
void launch_row_views(const int64_t *d_blk_row_off, const int32_t *d_blk_src_view, int n_blocks,
                      const int64_t *d_line_off, int vb, int n_views, int64_t *d_vrow, int32_t *d_vtile, int64_t *d_vtab,
                      cudaStream_t s);
cudaError_t launch_row_sort(const int32_t *d_pairs, const int64_t *d_blk_row_off, const int32_t *d_blk_ng_view,
                            const int64_t *d_blk_pair_off, int n_blocks, const int64_t *d_line_off, int vb,
                            const int64_t *d_vrow, const int32_t *d_vtile, const int64_t *d_vtab, int i_lo, int i_hi,
                            int tile0, int n_tiles, int max_lines, uint32_t *d_tab, uint32_t *d_node_row_off,
                            unsigned int *d_max_rows, uint32_t *d_key, uint32_t *d_val, int *d_err, cudaStream_t s);
void launch_extract_nvalid(const NodeRecord *nodes, int64_t node_begin, int64_t n, uint32_t *out, cudaStream_t s);
void launch_compact_edges_only(const uint8_t *row_state, const uint32_t *row_ng, const uint32_t *node_row_off,
                               const uint32_t *edge_off, int64_t node_begin, int64_t n, int ns, uint32_t *edge_ng,
                               cudaStream_t s);
void launch_edge_pairs(const uint32_t *edge_off, const uint32_t *edge_ng, const int64_t *line_off,
                       int64_t node_begin, int64_t n_nodes, int64_t n_edges, int64_t *out, cudaStream_t s);
void launch_edges_for_host(const uint32_t *edge_off, const uint32_t *edge_ng, const int32_t *img_ids,
                           int64_t n_nodes_shard, int64_t n_edges, int64_t node_begin, int64_t n_nodes_total,
                           int64_t *node_off, int32_t *pairs, cudaStream_t s);
void launch_zero_words(void *d_dst, int n_words, cudaStream_t s);
// one (source image, neighbour) match table as uploaded at TriangulateImage time
struct RawBlock {
  int32_t src_view, ng_view;
  int64_t n_rows;
  int64_t pair_off; // row offset into the device match store (-1: exhaustive)
  int32_t order, pad;
};
void launch_block_keys(const RawBlock *raw, int n_all, int vb, int ve, int exhaustive, uint32_t *key, uint32_t *val,
                       cudaStream_t s);
void launch_block_gather(const RawBlock *raw, const uint32_t *sorted_idx, int nb, int32_t *blk_src, int32_t *blk_ng,
                         int64_t *blk_pair_off, int64_t *blk_rows, cudaStream_t s);
void launch_edge_weights(const EdgeParams &p, cudaStream_t s);
void launch_gather_pack(const NodeRecord *nodes, int64_t node_begin, int64_t n_nodes, int64_t max_nodes,
                        const uint32_t *edge_off, const uint32_t *edge_ng, const int64_t *line_off, int64_t cap_edges,
                        char *msg, cudaStream_t s);
void launch_gather_unpack(const char *msgs, int world, const int64_t *rank_node_begin, int64_t max_nodes, int64_t cap_edges,
                          int64_t msg_bytes, NodeRecord *nodes, int64_t *edges, int64_t *scal, cudaStream_t s);

} // namespace lm
