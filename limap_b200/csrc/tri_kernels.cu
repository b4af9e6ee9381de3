// tri_kernels.cu — sm_100a kernels of the line-triangulation hot path.
//
//   tri_node_kernel : one CTA per 2D line ("node"). Fuses
//       BaseLineTriangulator::triangulateOneNode   (triangulation/base_line_triangulator.cc:161-337)
//       GlobalLineTriangulator::scoreOneNode       (triangulation/global_line_triangulator.cc:71-161)
//     so that the candidate set of a node lives only in shared memory: match rows are read once from
//     HBM, candidates are never written back unless debug_mode asks for them.
//   row_count / row_scan / row_scatter : turn the per-(image, neighbour) match tables into node-major rows (per-view
//       stable counting sort); expand_rows / node_offsets + a radix sort do it for views with many lines and for
//       exhaustive matching.
//   collect_edges / edge_weights : run_clustering's edge list and 3d scores
//       (global_line_triangulator.cc:234-291).
//
// Outputs and final decisions are fp64 (every gate of the reference is a hard threshold on a transcendental and
// the contract is bit-exact candidate indices); fp32 appears only in pruning gates with explicit margins
// (see DESIGN.md "Precision").
#include "tri_kernels.cuh"
#include <algorithm>
#include <cstdio>
#include <cub/block/block_scan.cuh>

namespace lm {

#ifndef LM_TRI_MIN_BLOCKS
#define LM_TRI_MIN_BLOCKS 4
#endif
static constexpr int kThreads = 128;
static constexpr int kWarps = kThreads / 32;
// per-candidate staging: 17 doubles (exact fp64 data + score), 11 floats (fp32 gate copies), ng + row
// (2 x uint32); plus two survivor lists per warp
// Staging the neighbour views of a node in shared memory with TMA bulk copies (cp.async.bulk + mbarrier) is
// implemented and parity-tested, and measured 3% SLOWER than the L1-cached generic loads it replaces on hypersim100
// (same box, 5 runs each: 6.90 ms with, 6.68 ms without; profiles/r02_tri_ab.txt): the views are already L1-resident
// (100 views x 208 B), so the copies only add a scan, two barriers per 128 rows and the mbarrier wait. Off by default
// for the headline instantiation; the VP instantiation (three proposals per row, each reading the neighbour view) keeps
// it on, which also keeps the path under the parity tests (test_vp_proposals, golden tri_vp_proposals).
#ifndef LM_TRI_TMA
#define LM_TRI_TMA 0
#endif
#ifndef LM_KFLUSH
#define LM_KFLUSH 64
#endif
static constexpr int kFlush = LM_KFLUSH;     // a warp flushes its survivor list once it holds this many pairs
static constexpr int kListExtra = kFlush + 32;
// per-candidate staging: 17 doubles (exact fp64 data + score), one 48-byte fp32 gate record, ng + row
// (2 x uint32); plus per warp two survivor lists (uint32) and one prefilter list (uint16)
static constexpr int kCandBytes = 17 * 8 + 48 + 8;

// Shared-memory staging per node. Generic layout: 17 doubles + 48-byte fp32 gate record + ng/row per candidate, two
// survivor lists and one prefilter list per warp. Fast layout (reduced-form scorer, plane-pair triangulation): 20 doubles
// (three reciprocals more), a 32-byte gate record, ng/row, the depth-sorted order (float key + uint16 index) per
// candidate, and per warp one pair list (uint16) with its scores (double): 246 bytes per candidate slot.
size_t tri_smem_bytes(int cap, bool fast) {
  if (fast) return (size_t)cap * (20 * 8 + kWarps * 8 + 32 + 8 + 4 + 2 + kWarps * 2);
  return (size_t)cap * kCandBytes + (size_t)kWarps * 2 * (cap + kListExtra) * 4 + (size_t)kWarps * cap * 2;
}
// Split scorer (tri_score_kernel): the fast layout without the four segment coordinates (a 4-byte global segment index
// instead) and without zs / ze / unc (read from the candidate records where phase C outputs them): 194 bytes per slot.
size_t tri_score_smem_bytes(int cap) { return (size_t)cap * (13 * 8 + kWarps * 8 + 32 + 12 + 4 + 2 + kWarps * 2); }

// fp32 copy of a candidate for the pruning gates (three 16-byte loads, conflict-free at 48-byte stride):
// unit direction, endpoints relative to the source camera centre, squared scale-invariance limits of the
// candidate taken as l_i.
struct __align__(16) GateRec {
  float dx, dy, dz, lims2;
  float sx, sy, sz, lime2;
  float ex, ey, ez, pad;
};

// Fast-path gate record. Every candidate of a node starts on the ray of the source line's start point and ends on the
// ray of its end point (X = ray * lambda + C1 in both the plane-pair and the VP-constrained triangulation), so the
// scale-invariant endpoint test of LineLinker3d (line_linker.cc:269-277) is an interval test on lambda: 1-D, sortable.
struct __align__(16) GateRecF {
  float dx, dy, dz, lam_e; // unit direction; distance of the end point along the end ray
  float lam_s;             // distance of the start point along the start ray
  float lim_s, lim_e;      // largest |delta lambda| that can still pass, taken as l_i (widened, see phase A)
  int img;                 // neighbour view of the candidate
};

struct Slab {
  double *sx, *sy, *sz, *ex, *ey, *ez, *dx, *dy, *dz, *zs, *ze, *unc, *q0, *q1, *q2, *q3, *score;
  double *izs2, *ize2, *inb; // fast layout only: 1/(zs+EPS)^2, 1/(ze+EPS)^2, 1/|q|^2
  GateRec *gate;
  uint32_t *ng, *row;
  uint32_t *list;            // [kWarps][2][cap + kListExtra]: (row << 16 | j) survivor entries
  uint16_t *list0;           // [kWarps][cap]: j of the start-point prefilter
  // fast layout only
  GateRecF *gatef;
  float *slam;               // [cap] lam_s in ascending order
  uint16_t *sidx;            // [cap] candidate of each sorted position
  double *psc;               // [kWarps][cap] scores of a warp's pair list
  uint16_t *pent;            // [kWarps][cap] j of a warp's pair list (rows contiguous)
  uint32_t *seg;             // split layout only: [cap] global segment index (into TriParams::segs) of the candidate
  LM_D void carve(char *base, int cap, bool fast) {
    seg = nullptr;
    if (fast) { carve_fast(base, cap); return; }
    gatef = nullptr; slam = nullptr; sidx = nullptr; psc = nullptr; pent = nullptr;
    double *d = reinterpret_cast<double *>(base);
    sx = d; sy = sx + cap; sz = sy + cap; ex = sz + cap; ey = ex + cap; ez = ey + cap;
    dx = ez + cap; dy = dx + cap; dz = dy + cap; zs = dz + cap; ze = zs + cap; unc = ze + cap;
    q0 = unc + cap; q1 = q0 + cap; q2 = q1 + cap; q3 = q2 + cap; score = q3 + cap;
    double *nx = score + cap;
    izs2 = ize2 = inb = nullptr;
    if (fast) { izs2 = nx; ize2 = izs2 + cap; inb = ize2 + cap; nx = inb + cap; }
    gate = reinterpret_cast<GateRec *>(nx);
    ng = reinterpret_cast<uint32_t *>(gate + cap);
    row = ng + cap;
    list = row + cap;
    list0 = reinterpret_cast<uint16_t *>(list + (size_t)kWarps * (fast ? 1 : 2) * (cap + kListExtra));
  }
  LM_D void carve_fast(char *base, int cap) {
    double *d = reinterpret_cast<double *>(base);
    sx = d; sy = sx + cap; sz = sy + cap; ex = sz + cap; ey = ex + cap; ez = ey + cap;
    dx = ez + cap; dy = dx + cap; dz = dy + cap; zs = dz + cap; ze = zs + cap; unc = ze + cap;
    q0 = unc + cap; q1 = q0 + cap; q2 = q1 + cap; q3 = q2 + cap; score = q3 + cap;
    izs2 = score + cap; ize2 = izs2 + cap; inb = ize2 + cap;
    psc = inb + cap;                                              // byte 160 cap
    gatef = reinterpret_cast<GateRecF *>(psc + (size_t)kWarps * cap); // byte 192 cap
    ng = reinterpret_cast<uint32_t *>(gatef + cap);               // byte 224 cap
    row = ng + cap;
    slam = reinterpret_cast<float *>(row + cap);                  // byte 232 cap
    sidx = reinterpret_cast<uint16_t *>(slam + cap);              // byte 236 cap
    pent = sidx + cap;                                            // byte 238 cap, [kWarps][cap]
    gate = nullptr; list = nullptr; list0 = nullptr; seg = nullptr;
  }
  // tri_score_kernel: tri_score_smem_bytes() per slot, no zs / ze / unc / q0..q3
  LM_D void carve_split(char *base, int cap) {
    double *d = reinterpret_cast<double *>(base);
    sx = d; sy = sx + cap; sz = sy + cap; ex = sz + cap; ey = ex + cap; ez = ey + cap;
    dx = ez + cap; dy = dx + cap; dz = dy + cap; score = dz + cap;
    izs2 = score + cap; ize2 = izs2 + cap; inb = ize2 + cap;
    psc = inb + cap;                                              // byte 104 cap
    gatef = reinterpret_cast<GateRecF *>(psc + (size_t)kWarps * cap); // byte 136 cap (cap is a multiple of 32)
    ng = reinterpret_cast<uint32_t *>(gatef + cap);               // byte 168 cap
    row = ng + cap;
    seg = row + cap;
    slam = reinterpret_cast<float *>(seg + cap);                  // byte 180 cap
    sidx = reinterpret_cast<uint16_t *>(slam + cap);              // byte 184 cap
    pent = sidx + cap;                                            // byte 186 cap, [kWarps][cap]
    zs = ze = unc = q0 = q1 = q2 = q3 = nullptr;
    gate = nullptr; list = nullptr; list0 = nullptr;
  }
};

// ---- TMA bulk copies (cp.async.bulk + mbarrier): the neighbour views of a node are staged in shared memory ----------
LM_D uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
LM_D void mbar_init(unsigned long long *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
LM_D void mbar_arrive_expect_tx(unsigned long long *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
LM_D void bulk_copy_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
LM_D void mbar_wait(unsigned long long *bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
  }
}

struct Cand {
  vec3<double> s, e;
  double zs, ze, unc;
  double lam_s, lam_e; // s = ray1s * lam_s + C1, e = ray1e * lam_e + C1 (not set by endpoint triangulation)
};

LM_D double4 ld_seg(const double4 *p) {
  const double2 a = __ldg(reinterpret_cast<const double2 *>(p));
  const double2 b = __ldg(reinterpret_cast<const double2 *>(p) + 1);
  return make_double4(a.x, a.y, b.x, b.y);
}
LM_D double deg_from_cos_abs(double c) { return acos(fabs(c)) * consts<double>::rad2deg(); }

// triangulate_point (triangulation/functions.cc:100-117): mid-point method, 2x2 LDLT.
LM_D bool triangulate_point(const ViewD &v1, const ViewD &v2, vec3<double> n1e, vec3<double> n2e, vec3<double> C1,
                            vec3<double> C2, vec3<double> &out) {
  double a00 = dot(n1e, n1e), a01 = -dot(n1e, n2e), a10 = -dot(n2e, n1e), a11 = dot(n2e, n2e);
  double b0 = dot(n1e, C2 - C1), b1 = dot(n2e, C1 - C2);
  double r0, r1;
  if (a00 >= a11) {
    double l10 = a10 / a00, d1 = a11 - l10 * a01, y1 = b1 - l10 * b0;
    r1 = y1 / d1;
    r0 = (b0 - a01 * r1) / a00;
  } else {
    double l01 = a01 / a11, d0 = a00 - l01 * a10, y0 = b0 - l01 * b1;
    r0 = y0 / d0;
    r1 = (b1 - a10 * r0) / a11;
  }
  out = (n1e * r0 + C1 + n2e * r1 + C2) * 0.5;
  double z1 = v1.P[8] * out.x + v1.P[9] * out.y + v1.P[10] * out.z + v1.P[11];
  double z2 = v2.P[8] * out.x + v2.P[9] * out.y + v2.P[10] * out.z + v2.P[11];
  return !(z1 < consts<double>::eps() || z2 < consts<double>::eps());
}

// Per-node constants of the source line (computed redundantly by every thread: ~60 flops).
struct Src {
  double4 l1;
  vec3<double> w1s, w1e;     // M1 [p;1] (unnormalised world rays)
  vec3<double> ray1s, ray1e; // normalised
  vec3<double> C1;
  vec3<double> n1;           // getNormalDirection(l1, view1) (only for VP proposals)
  bool ok;
};

// Margin comparison of squared quantities: returns +1 / -1 when lhs is above / below rhs by more than
// 1e-9 relative (far beyond fp64 rounding of these short expressions), 0 when too close to call -- the
// caller then evaluates the reference's transcendental form for that single test.
LM_D int cmp_margin(double lhs, double rhs) {
  const double REL = 1e-9;
  if (lhs > rhs * (1.0 + REL)) return 1;
  if (lhs < rhs * (1.0 - REL)) return -1;
  return 0;
}

// Line3d::sensitivity(view) > th  (base/linebase.cc:100-107), decided without acos when clear:
// 90 - acos|c| > th  <=>  |c| > sin(th).
LM_D bool sensitivity_exceeds(const TriParams &p, const ViewD &v, vec3<double> Xs, vec3<double> Xe, vec3<double> dir_raw) {
  const vec3<double> hs = proj_h(v.P, Xs), he = proj_h(v.P, Xe);
  const double is = 1.0 / (hs.z + consts<double>::eps()), ie = 1.0 / (he.z + consts<double>::eps());
  const vec2<double> mid = mk2((hs.x * is + he.x * ie) * 0.5, (hs.y * is + he.y * ie) * 0.5);
  const vec3<double> d3 = mat3_mul_h(v.M, mid.x, mid.y);
  const double t = dot(dir_raw, d3);
  const int cm = cmp_margin(t * t, p.sin2_sens * dot(dir_raw, dir_raw) * dot(d3, d3));
  if (cm != 0 && p.sens_poly_ok) return cm > 0;
  return 90.0 - deg_from_cos_abs(dot(normalized(dir_raw), normalized(d3))) > p.sensitivity_threshold;
}

// One match row -> candidate. Steps follow triangulateOneNode "Step 3" (base_line_triangulator.cc:290-326).
// Unit-vector normalisations that do not change a decision or an output beyond rounding are dropped; the
// angle / sensitivity gates use margin forms with the reference's acos form as the tie fallback.
// The gates of a match row that need no 3D point: segment length, ray-plane angles, epipolar IoU (:290-305).
LM_D bool cand_gates(const TriParams &p, const ViewD &v2, const Src &src, const double4 &l2) {
  const vec2<double> s2 = mk2(l2.x, l2.y), e2 = mk2(l2.z, l2.w);
  const vec2<double> v2d = e2 - s2;
  const double len2sq = dot(v2d, v2d);
  { // |l2| <= min_length_2d (:177), squared with an exact tie fallback
    const double m2 = p.min_length_2d * p.min_length_2d;
    if (p.min_length_2d >= 0.0) {
      if (len2sq <= m2 * (1.0 - 1e-12)) return false;
      if (len2sq < m2 * (1.0 + 1e-12) && sqrt(len2sq) <= p.min_length_2d) return false;
    }
  }
  if (p.disable_algebraic) return false;
  const vec3<double> c2s = mat3_mul_h(v2.M, l2.x, l2.y);
  const vec3<double> c2e = mat3_mul_h(v2.M, l2.z, l2.w);
  // getNormalDirection (functions.cc:28-35) + ray-plane angle tests (:292-302):
  // 90 - acos|n2.ray| < th  <=>  |n2.ray| < sin(th)
  {
    const vec3<double> n2 = cross(c2s, c2e);
    const double nn = dot(n2, n2);
    const double ts = dot(n2, src.ray1s), te = dot(n2, src.ray1e);
    int cs_ = cmp_margin(ts * ts, p.sin2_tri * nn), ce_ = cmp_margin(te * te, p.sin2_tri * nn);
    if (!p.tri_poly_ok) cs_ = ce_ = 0;
    if (cs_ < 0 || ce_ < 0) return false; // one endpoint ray clearly below the threshold
    if (cs_ == 0 || ce_ == 0) {           // too close to call: the reference's acos form decides
      const vec3<double> n2u = normalized(n2);
      if (cs_ == 0 && 90.0 - deg_from_cos_abs(dot(n2u, src.ray1s)) < p.line_tri_angle_threshold) return false;
      if (ce_ == 0 && 90.0 - deg_from_cos_abs(dot(n2u, src.ray1e)) < p.line_tri_angle_threshold) return false;
    }
  }
  const vec3<double> C2 = mk3(v2.C[0], v2.C[1], v2.C[2]);
  // compute_epipolar_IoU (functions.cc:76-98). F x1 = M2^T ((C1 - C2) x (M1 x1)) exactly
  // (F = K2^-T [t]x R2 R1^T K1^-1 with t = R2 (C1 - C2)); dehomogeneous() of the cross product of two
  // normalised line vectors == raw.xy / (raw.z + EPS |a| |b|).
  {
    const vec3<double> base = src.C1 - C2;
    const vec3<double> l2h = cross(mk3(l2.x, l2.y, 1.0), mk3(l2.z, l2.w, 1.0));
    const double nl2 = dot(l2h, l2h);
    const vec3<double> eps_ = mat3T_mul(v2.M, cross(base, src.w1s));
    const vec3<double> hs = cross(l2h, eps_);
    const double ws = 1.0 / (hs.z + consts<double>::eps() * sqrt(nl2 * dot(eps_, eps_)));
    const vec3<double> epe_ = mat3T_mul(v2.M, cross(base, src.w1e));
    const vec3<double> he = cross(l2h, epe_);
    const double we = 1.0 / (he.z + consts<double>::eps() * sqrt(nl2 * dot(epe_, epe_)));
    const vec2<double> cs = mk2(hs.x * ws, hs.y * ws), ce = mk2(he.x * we, he.y * we);
    const double il2 = 1.0 / len2sq;
    double c1 = dot(cs - s2, v2d) * il2;
    double c2 = dot(ce - s2, v2d) * il2;
    if (c1 > c2) { double t = c1; c1 = c2; c2 = t; }
    double IoU = (smin(c2, 1.0) - smax(c1, 0.0)) / (smax(c2, 1.0) - smin(c1, 0.0));
    if (fabs(IoU - p.IoU_threshold) < 1e-7) {
      // too close to the threshold: evaluate in the reference's normalised form
      const vec3<double> coor_l2 = normalized(l2h);
      const vec2<double> cs2 = dehom(cross(coor_l2, normalized(eps_)));
      const vec2<double> ce2 = dehom(cross(coor_l2, normalized(epe_)));
      const vec2<double> dir2 = normalized(v2d);
      const double len2 = norm(s2 - e2);
      c1 = dot(cs2 - s2, dir2) / len2;
      c2 = dot(ce2 - s2, dir2) / len2;
      if (c1 > c2) { double t = c1; c1 = c2; c2 = t; }
      IoU = (smin(c2, 1.0) - smax(c1, 0.0)) / (smax(c2, 1.0) - smin(c1, 0.0));
    }
    if (IoU < p.IoU_threshold) return false;
  }
  return true;
}

// Triangulation of a row that passed cand_gates, with the gates on the 3D points (:306-326).
template <bool ALLOW_ENDP>
LM_D bool cand_triangulate(const TriParams &p, const ViewD &v1, const ViewD &v2, const Src &src, const double4 &l2, Cand &c) {
  const vec3<double> c2s = mat3_mul_h(v2.M, l2.x, l2.y);
  const vec3<double> c2e = mat3_mul_h(v2.M, l2.z, l2.w);
  const vec3<double> C2 = mk3(v2.C[0], v2.C[1], v2.C[2]);
  vec3<double> Xs, Xe;
  const double EPS = consts<double>::eps();
  if (!ALLOW_ENDP || !p.use_endpoints_triangulation) {
    // line_triangulation (functions.cc:194-233): plane-pair intersection. Only lambda_0 is used, which
    // does not depend on the norms of the second and third column.
    const vec3<double> B = C2 - src.C1;
    const vec3<double> nb = mk3(-c2s.x, -c2s.y, -c2s.z), nc = mk3(-c2e.x, -c2e.y, -c2e.z);
    const vec3<double> ls = solve3_cols(src.ray1s, nb, nc, B);
    Xs = src.ray1s * ls.x + src.C1;
    const vec3<double> le = solve3_cols(src.ray1e, nb, nc, B);
    Xe = src.ray1e * le.x + src.C1;
    c.lam_s = ls.x;
    c.lam_e = le.x;
    c.zs = v1.P[8] * Xs.x + v1.P[9] * Xs.y + v1.P[10] * Xs.z + v1.P[11];
    c.ze = v1.P[8] * Xe.x + v1.P[9] * Xe.y + v1.P[10] * Xe.z + v1.P[11];
    if (c.zs < EPS || c.ze < EPS) return false;
    const double d21 = v2.P[8] * Xs.x + v2.P[9] * Xs.y + v2.P[10] * Xs.z + v2.P[11];
    const double d22 = v2.P[8] * Xe.x + v2.P[9] * Xe.y + v2.P[10] * Xe.z + v2.P[11];
    if (d21 < EPS || d22 < EPS) return false;
    if (isnan(Xs.x) || isnan(Xe.x)) return false;
  } else {
    // triangulate_line_by_endpoints (functions.cc:172-190)
    const vec3<double> r2s = normalized(c2s), r2e = normalized(c2e);
    if (!triangulate_point(v1, v2, src.ray1s, r2s, src.C1, C2, Xs)) return false;
    if (!triangulate_point(v1, v2, src.ray1e, r2e, src.C1, C2, Xe)) return false;
    c.zs = v1.P[8] * Xs.x + v1.P[9] * Xs.y + v1.P[10] * Xs.z + v1.P[11];
    c.ze = v1.P[8] * Xe.x + v1.P[9] * Xe.y + v1.P[10] * Xe.z + v1.P[11];
    c.lam_s = c.lam_e = 0.0;
  }
  // sensitivity in both views (:315-317)
  const vec3<double> dir_raw = Xe - Xs;
  if (sensitivity_exceeds(p, v1, Xs, Xe, dir_raw) && sensitivity_exceeds(p, v2, Xs, Xe, dir_raw)) return false;
  // uncertainty = min(u1, u2) (:319-321; linebase.cc:109-116; camera.cc:228-242)
  {
    const double d1 = (c.zs + c.ze) / 2.0;
    const double u1 = p.var2d * d1 / v1.fbar;
    const double z2s = v2.P[8] * Xs.x + v2.P[9] * Xs.y + v2.P[10] * Xs.z + v2.P[11];
    const double z2e = v2.P[8] * Xe.x + v2.P[9] * Xe.y + v2.P[10] * Xe.z + v2.P[11];
    const double u2 = p.var2d * ((z2s + z2e) / 2.0) / v2.fbar;
    c.unc = smin(u1, u2);
  }
  // test_line_inside_ranges (functions.cc:8-26)
  if (p.ranges_flag) {
    if (Xs.x < p.rlo[0] || Xs.x > p.rhi[0] || Xs.y < p.rlo[1] || Xs.y > p.rhi[1] || Xs.z < p.rlo[2] || Xs.z > p.rhi[2])
      return false;
    if (Xe.x < p.rlo[0] || Xe.x > p.rhi[0] || Xe.y < p.rlo[1] || Xe.y > p.rhi[1] || Xe.z < p.rlo[2] || Xe.z > p.rhi[2])
      return false;
  }
  c.s = Xs;
  c.e = Xe;
  return true;
}

template <bool ALLOW_ENDP>
LM_D bool gen_candidate(const TriParams &p, const ViewD &v1, const ViewD &v2, const Src &src, uint32_t ngv, uint32_t ngl,
                        Cand &c, double4 &l2out) {
  const double4 l2 = ld_seg(&p.segs[p.line_off[ngv] + ngl]);
  l2out = l2;
  return cand_gates(p, v2, src, l2) && cand_triangulate<ALLOW_ENDP>(p, v1, v2, src, l2, c);
}

// triangulate_line_with_direction (triangulation/functions.cc:389-446) for a VP proposal
// (base_line_triangulator.cc:258-288): fp64, formulas as in the reference (this path is off by default).
// `direction` is the unit world direction of the VP seen from view 1.
LM_D bool gen_vp_candidate(const TriParams &p, const ViewD &v1, const ViewD &v2, const Src &src, vec3<double> c2s,
                           vec3<double> c2e, vec3<double> direction, Cand &c) {
  const double EPS = consts<double>::eps();
  const vec3<double> n1 = src.n1;
  vec3<double> direc = direction - n1 * dot(n1, direction);
  if (norm(direc) < EPS) return false;
  direc = normalized(direc);
  const vec3<double> perp = cross(n1, direc);
  double a1s = dot(src.ray1s, perp), a1e = dot(src.ray1e, perp);
  if (a1s < 0) { a1s *= -1; a1e *= -1; }
  if (a1s < 0.001 || a1e < 0.001) return false; // MIN_VALUE
  const vec3<double> C2 = mk3(v2.C[0], v2.C[1], v2.C[2]);
  const vec3<double> n2 = normalized(cross(c2s, c2e));
  const double c1s = dot(n2, src.ray1s), c1e = dot(n2, src.ray1e), b = dot(n2, C2 - src.C1);
  const double c1 = c1s, c2 = c1e * a1s / a1e;
  const double d1s = (c1 + c2) * b / (c1 * c1 + c2 * c2);
  const double d1e = d1s * a1s / a1e;
  const vec3<double> Xs = src.ray1s * d1s + src.C1, Xe = src.ray1e * d1e + src.C1;
  c.lam_s = d1s;
  c.lam_e = d1e;
  c.zs = v1.P[8] * Xs.x + v1.P[9] * Xs.y + v1.P[10] * Xs.z + v1.P[11];
  c.ze = v1.P[8] * Xe.x + v1.P[9] * Xe.y + v1.P[10] * Xe.z + v1.P[11];
  if (c.zs < EPS || c.ze < EPS) return false;
  const double z2s = v2.P[8] * Xs.x + v2.P[9] * Xs.y + v2.P[10] * Xs.z + v2.P[11];
  const double z2e = v2.P[8] * Xe.x + v2.P[9] * Xe.y + v2.P[10] * Xe.z + v2.P[11];
  if (z2s < EPS || z2e < EPS) return false;
  if (isnan(Xs.x) || isnan(Xe.x)) return false;
  const double u1 = p.var2d * ((c.zs + c.ze) / 2.0) / v1.fbar;
  const double u2 = p.var2d * ((z2s + z2e) / 2.0) / v2.fbar;
  c.unc = smin(u1, u2);
  if (p.ranges_flag) {
    if (Xs.x < p.rlo[0] || Xs.x > p.rhi[0] || Xs.y < p.rlo[1] || Xs.y > p.rhi[1] || Xs.z < p.rlo[2] || Xs.z > p.rhi[2])
      return false;
    if (Xe.x < p.rlo[0] || Xe.x > p.rhi[0] || Xe.y < p.rlo[1] || Xe.y > p.rhi[1] || Xe.z < p.rlo[2] || Xe.z > p.rhi[2])
      return false;
  }
  c.s = Xs;
  c.e = Xe;
  return true;
}

// Pair score of candidates (i, j) of one node (global_line_triangulator.cc:91-104):
// min(LineLinker3d::compute_score(l_i, l_j), LineLinker2d::compute_score(proj_{view j}(l_i), seg_j)),
// 0 when either is 0.
LM_D double pair_score(const TriParams &p, const seg<vec3<double>> &Li, vec3<double> di, double zsi, double zei,
                       const Slab &sl, int j, uint32_t vj) {
  // 3d: angle (line_linker.cc:185-192) then scale-invariant endpoint distance (:269-277)
  const LinkerDev<double> &c3 = p.l3d;
  double score3 = 1.0;
  {
    double cs = fabs(di.x * sl.dx[j] + di.y * sl.dy[j] + di.z * sl.dz[j]);
    double angle = acos(cs) * consts<double>::rad2deg();
    score3 = smin(score3, thresh0(expscore(angle, c3.th_angle * c3.mult), c3.score_th));
    if (score3 < c3.score_th) return 0.0;
    vec3<double> sj = mk3(sl.sx[j], sl.sy[j], sl.sz[j]), ej = mk3(sl.ex[j], sl.ey[j], sl.ez[j]);
    double ds = norm(Li.s - sj), de = norm(Li.e - ej);
    double dist = smax(ds / (zsi + consts<double>::eps()), de / (zei + consts<double>::eps()));
    score3 = smin(score3, thresh0(expscore(dist, c3.th_scaleinv * c3.mult), c3.score_th));
    if (score3 == 0.0) return 0.0;
  }
  // 2d: project l_i into the view of candidate j (linebase.cc:93-98) and score against its 2D segment
  const ViewD &v = p.views[vj];
  seg<vec2<double>> a, b;
  a.s = dehom(proj_h(v.P, Li.s));
  a.e = dehom(proj_h(v.P, Li.e));
  b.s = mk2(sl.q0[j], sl.q1[j]);
  b.e = mk2(sl.q2[j], sl.q3[j]);
  double score2 = linker_score<double, vec2<double>>(p.l2d, a, b, 1.0, false, 0.0, 0.0);
  if (score2 == 0.0) return 0.0;
  return smin(score3, score2);
}

// The same pair score in algebraically reduced form (used unless innerseg is enabled on the 2d linker):
// every sub-score of the two linkers is exp(-q_k/2) with q_k = (v_k/sigma_k)^2 zeroed below score_th, and
// their minimum is exp(-max_k q_k / 2) because exp is monotone -- one exp instead of up to six; distances
// enter as squares (no square roots: (d/sigma)^2 = d^2/sigma^2, max of the four perpendicular distances =
// sqrt of the max of their squares), directions are never normalised (|cos| = |a.b|/sqrt(|a|^2|b|^2)) and
// homogeneous divisions use one reciprocal. NaN angles are ignored exactly like std::min ignores a NaN
// sub-score (line_dists.h:62-66). Polynomial early-outs skip the transcendental part for clear failures.
// asin(sqrt(t))^2 / t for 0 <= t <= 1/16 (angles up to 14.4 deg): asin^2(x) = sum_n 2^(2n-1) x^(2n) / (n^2 C(2n,n));
// 14 terms leave a relative remainder below 3e-19.
LM_D double asin2_over_t(double t) {
  double r = 0.017069849551821746;
  r = fma(r, t, 0.019089950090498877);
  r = fma(r, t, 0.02154247840073658);
  r = fma(r, t, 0.02456910759753428);
  r = fma(r, t, 0.028377319275152094);
  r = fma(r, t, 0.03328204112517838);
  r = fma(r, t, 0.03978243978243978);
  r = fma(r, t, 0.04871319157033443);
  r = fma(r, t, 0.06156806156806157);
  r = fma(r, t, 0.08126984126984127);
  r = fma(r, t, 0.11428571428571428);
  r = fma(r, t, 0.17777777777777778);
  r = fma(r, t, 0.3333333333333333);
  r = fma(r, t, 1.0);
  return r;
}
// squared angle in degrees between two directions from sin^2 = t (t <= 1/16) or from |cos| otherwise
LM_D double angle2_deg(double t, double abs_cos) {
  const double k = consts<double>::rad2deg();
  if (t <= 0.0625) return t * asin2_over_t(t) * (k * k);
  const double a = acos(abs_cos) * k;
  return a * a;
}

// Reduced-form pair score: same value as pair_score() up to rounding. min over sub-scores of exp(-(v/sigma)^2/2)
// == exp(-max (v/sigma)^2 / 2), so the squared normalised deviations are maximised and one exponential is taken;
// angles come from sin^2 (cross products) through the asin^2 series, distances stay squared, and the divisors
// that depend on one candidate only (depths of l_i, |q_j|^2) are reciprocals prepared in phase A.
template <bool SPLIT = false>
LM_D double pair_score_fast(const TriParams &p, const Slab &sl, int i, int j, uint32_t vj) {
  const double EPS = consts<double>::eps();
  const LinkerDev<double> &c3 = p.l3d;
  const LinkerDev<double> &c2 = p.l2d;
  const vec3<double> si = mk3(sl.sx[i], sl.sy[i], sl.sz[i]), ei = mk3(sl.ex[i], sl.ey[i], sl.ez[i]);
  double Q = 0.0; // running maximum of the squared normalised deviations
  // ---- 3d: angle (line_linker.cc:185-192) + scale-invariant endpoint distance (:269-277)
  {
    const vec3<double> di = mk3(sl.dx[i], sl.dy[i], sl.dz[i]), dj = mk3(sl.dx[j], sl.dy[j], sl.dz[j]);
    // products rounded separately: cross(di, dj) == -cross(dj, di) bit for bit, so two candidates that support
    // only each other through the angle term tie exactly, as they do with the reference's symmetric acos(|di.dj|)
    const vec3<double> cr = mk3(__dmul_rn(di.y, dj.z) - __dmul_rn(di.z, dj.y), __dmul_rn(di.z, dj.x) - __dmul_rn(di.x, dj.z),
                                __dmul_rn(di.x, dj.y) - __dmul_rn(di.y, dj.x));
    double a2 = angle2_deg(dot(cr, cr), fabs(dot(di, dj)));
    if (!(dot(di, di) * dot(dj, dj) > 0.5)) a2 = 8100.0; // zero-length candidate: acos(0) = 90 deg
    if (a2 == a2) Q = a2 * (p.inv_sig_a3 * p.inv_sig_a3);
    const vec3<double> ds = si - mk3(sl.sx[j], sl.sy[j], sl.sz[j]), de = ei - mk3(sl.ex[j], sl.ey[j], sl.ez[j]);
    const double r2 = fmax(dot(ds, ds) * sl.izs2[i], dot(de, de) * sl.ize2[i]);
    Q = fmax(Q, r2 * p.inv_sig_s3 * p.inv_sig_s3);
    if (Q > p.q_cut3) return 0.0; // some 3d sub-score is clearly below score_th
  }
  // ---- 2d: projection of l_i into the view of candidate j (linebase.cc:93-98)
  const ViewD &v = p.views[vj];
  const vec3<double> hs = proj_h(v.P, si), he = proj_h(v.P, ei);
  const double ws = 1.0 / (hs.z + EPS), we = 1.0 / (he.z + EPS);
  const vec2<double> as = mk2(hs.x * ws, hs.y * ws), ae = mk2(he.x * we, he.y * we);
  vec2<double> bs, be;
  if constexpr (SPLIT) { // the split scorer keeps the global segment index of a candidate instead of its four coordinates
    const double4 q = ld_seg(&p.segs[sl.seg[j]]);
    bs = mk2(q.x, q.y);
    be = mk2(q.z, q.w);
  } else {
    bs = mk2(sl.q0[j], sl.q1[j]);
    be = mk2(sl.q2[j], sl.q3[j]);
  }
  const vec2<double> va = ae - as, vb = be - bs;
  const double na2 = dot(va, va), nb2 = dot(vb, vb);
  const double dab = dot(va, vb);
  const double ina = 1.0 / na2, inb = sl.inb[j];
  double Q2 = 0.0;
  double ang2 = 0.0; // squared 2d angle in degrees
  if (c2.use_angle) {
    if (dab * dab < p.cos2_th2d * na2 * nb2 * (1.0 - 1e-9)) return 0.0; // |cos| clearly below cos(th_angle)
    if (na2 > 0.0 && nb2 > 0.0) {
      const double cr = va.x * vb.y - va.y * vb.x;
      const double t = cr * cr * (ina * inb);
      ang2 = angle2_deg(t, (t <= 0.0625) ? 0.0 : fabs(dab) / sqrt(na2 * nb2));
    } else {
      ang2 = 8100.0; // acos(0) = 90 deg
    }
    if (ang2 == ang2) Q2 = ang2 * (p.inv_sig_a2 * p.inv_sig_a2);
  }
  double bio = 0.0;
  if (c2.use_overlap) { // compute_bioverlap (line_dists.h:190-208)
    double p1 = dot(as - bs, vb) * inb, p2 = dot(ae - bs, vb) * inb;
    if (p1 > p2) { const double t = p1; p1 = p2; p2 = t; }
    const double o1 = smin(p2, 1.0) - smax(p1, 0.0);
    double r1 = dot(bs - as, va) * ina, r2 = dot(be - as, va) * ina;
    if (r1 > r2) { const double t = r1; r1 = r2; r2 = t; }
    const double o2 = smin(r2, 1.0) - smax(r1, 0.0);
    bio = smax(o1, o2);
    if (!(bio > c2.th_overlap)) return 0.0;
  }
  if (c2.use_angle && c2.use_overlap && c2.use_smartangle && bio < c2.th_smartoverlap) { // line_linker.cc:49-65
    double ratio = (c2.th_smartoverlap - bio) * p.inv_smart_den2;
    ratio = smin(ratio, 1.0);
    const double sig = (c2.th_angle - ratio * (c2.th_angle - c2.th_smartangle)) * c2.mult;
    if (ang2 == ang2) Q2 = fmax(Q2, ang2 / (sig * sig));
  }
  if (c2.use_perp) { // max of the four endpoint-to-infinite-line distances, squared (line_dists.h:105-133)
    const vec2<double> d0 = as - bs, d1 = ae - bs, d2 = bs - as, d3 = be - as;
    const double t0 = dot(d0, vb), t1 = dot(d1, vb), t2 = dot(d2, va), t3 = dot(d3, va);
    double m = fmax(dot(d0, d0) - t0 * t0 * inb, 0.0);
    m = fmax(m, dot(d1, d1) - t1 * t1 * inb);
    m = fmax(m, dot(d2, d2) - t2 * t2 * ina);
    m = fmax(m, dot(d3, d3) - t3 * t3 * ina);
    Q2 = fmax(Q2, m * p.inv_sig_p2 * p.inv_sig_p2);
  }
  // each linker applies its own score_th: exp(-Q/2) >= th <=> Q <= -2 ln th. Clear of both cuts by 1e-9 relative,
  // one exponential of the larger deviation is the score; next to a cut the two exponentials decide.
  if (Q2 > p.q_cut2) return 0.0;
  if (Q < p.q_cut3_lo && Q2 < p.q_cut2_lo) return exp(-fmax(Q, Q2) * 0.5);
  const double e3 = exp(-Q * 0.5), e2 = exp(-Q2 * 0.5);
  if (e3 < c3.score_th || e2 < c2.score_th) return 0.0;
  return smin(e3, e2);
}

// ---- pruning gates -----------------------------------------------------------------------------------
// The reference decides every sub-test on exp(-(v/sigma)^2/2) >= score_th, i.e. v <= th. The gates below
// only discard pairs that fail a sub-test by a margin far above the arithmetic error of the gate (fp32
// for the 3d tests, fp64 polynomial forms for the 2d tests); every surviving pair is then scored by
// pair_score(), which evaluates the reference formulas in fp64 and takes all decisions itself. Pruned
// pairs would have scored exactly 0, so results do not depend on the gates.

// 3d gate, fp32: angle (line_linker.cc:185-192) and scale-invariant endpoint distance (:269-277).
LM_D bool gate3d(const GateRec &r, const GateRec *g, float cos_th) {
  const float4 a = *reinterpret_cast<const float4 *>(&g->dx);
  const float cs = fabsf(r.dx * a.x + r.dy * a.y + r.dz * a.z);
  if (cs < cos_th) return false;
  const float4 b = *reinterpret_cast<const float4 *>(&g->sx);
  const float ax = r.sx - b.x, ay = r.sy - b.y, az = r.sz - b.z;
  if (ax * ax + ay * ay + az * az > r.lims2) return false;
  const float4 c = *reinterpret_cast<const float4 *>(&g->ex);
  const float bx = r.ex - c.x, by = r.ey - c.y, bz = r.ez - c.z;
  return !(bx * bx + by * by + bz * bz > r.lime2);
}

// gate3d without the start-point test (done by the prefilter)
LM_D bool gate3d_rest(const GateRec &r, const GateRec *g, float cos_th) {
  const float4 a = *reinterpret_cast<const float4 *>(&g->dx);
  if (fabsf(r.dx * a.x + r.dy * a.y + r.dz * a.z) < cos_th) return false;
  const float4 c = *reinterpret_cast<const float4 *>(&g->ex);
  const float bx = r.ex - c.x, by = r.ey - c.y, bz = r.ez - c.z;
  return !(bx * bx + by * by + bz * bz > r.lime2);
}

// 2d gate, fp64 without transcendentals: angle, overlap and perpendicular tests of
// LineLinker2d::compute_score (line_linker.cc:139-160) in margin form.
LM_D bool gate2d(const TriParams &p, const seg<vec3<double>> &Li, const Slab &sl, int j, uint32_t vj) {
  const LinkerDev<double> &c = p.l2d;
  const ViewD &v = p.views[vj];
  const vec2<double> as = dehom(proj_h(v.P, Li.s)), ae = dehom(proj_h(v.P, Li.e));
  const vec2<double> bs = mk2(sl.q0[j], sl.q1[j]), be = mk2(sl.q2[j], sl.q3[j]);
  const vec2<double> va = ae - as, vb = be - bs;
  const double na2 = dot(va, va), nb2 = dot(vb, vb);
  const double REL = 1e-9;
  if (c.use_angle) {
    const double d = dot(va, vb);
    if (d * d < p.cos2_th2d * na2 * nb2 * (1.0 - REL)) return false; // |cos| < cos(th_angle)
  }
  if (c.use_overlap) {
    // compute_bioverlap (line_dists.h:190-208) with p = dot / |l2|^2 (no normalisation)
    double p1 = dot(as - bs, vb) / nb2, p2 = dot(ae - bs, vb) / nb2;
    if (p1 > p2) { const double t = p1; p1 = p2; p2 = t; }
    const double o1 = smin(p2, 1.0) - smax(p1, 0.0);
    double r1 = dot(bs - as, va) / na2, r2 = dot(be - as, va) / na2;
    if (r1 > r2) { const double t = r1; r1 = r2; r2 = t; }
    const double o2 = smin(r2, 1.0) - smax(r1, 0.0);
    const double bio = smax(o1, o2);
    if (bio < c.th_overlap - REL * (1.0 + fabs(c.th_overlap))) return false;
  }
  if (c.use_perp) {
    // squared endpoint-to-infinite-line distances (line_dists.h:105-133)
    const vec2<double> d0 = as - bs, d1 = ae - bs, d2 = bs - as, d3 = be - as;
    const double t0 = dot(d0, vb), t1 = dot(d1, vb), t2 = dot(d2, va), t3 = dot(d3, va);
    double m = dot(d0, d0) - t0 * t0 / nb2;
    m = fmax(m, dot(d1, d1) - t1 * t1 / nb2);
    m = fmax(m, dot(d2, d2) - t2 * t2 / na2);
    m = fmax(m, dot(d3, d3) - t3 * t3 / na2);
    if (m > p.th_perp2_2d * (1.0 + REL) + REL) return false;
  }
  return true;
}

// ---- phases shared by the fused kernel and the split generate / score kernels ---------------------------------------
// Staging of one candidate in the scorer's shared-memory layout: the direction, the three reciprocals of the reduced-form
// scorer and the fp32 gate record (FAST) or the generic gate copy. SPLIT keeps the global segment index `segi` instead
// of the segment coordinates and leaves zs / ze / unc in the candidate record.
template <bool FAST, bool SPLIT>
LM_D void stage_cand(const TriParams &p, const Slab &sl, int idx, const Cand &c, double4 l2, uint32_t ng, uint32_t row,
                     vec3<double> C1, uint32_t segi = 0) {
  const vec3<double> dr = c.e - c.s;
  const double dn2 = dot(dr, dr);
  const vec3<double> d = (dn2 > 0.0) ? dr * (1.0 / sqrt(dn2)) : dr;
  sl.sx[idx] = c.s.x; sl.sy[idx] = c.s.y; sl.sz[idx] = c.s.z;
  sl.ex[idx] = c.e.x; sl.ey[idx] = c.e.y; sl.ez[idx] = c.e.z;
  sl.dx[idx] = d.x; sl.dy[idx] = d.y; sl.dz[idx] = d.z;
  if constexpr (SPLIT) {
    sl.seg[idx] = segi; // zs / ze / unc stay in the candidate record
  } else {
    sl.zs[idx] = c.zs; sl.ze[idx] = c.ze; sl.unc[idx] = c.unc;
    sl.q0[idx] = l2.x; sl.q1[idx] = l2.y; sl.q2[idx] = l2.z; sl.q3[idx] = l2.w;
  }
  if (FAST) {
    const double zs1 = c.zs + consts<double>::eps(), ze1 = c.ze + consts<double>::eps();
    const double qx = l2.z - l2.x, qy = l2.w - l2.y;
    sl.izs2[idx] = 1.0 / (zs1 * zs1); sl.ize2[idx] = 1.0 / (ze1 * ze1); sl.inb[idx] = 1.0 / (qx * qx + qy * qy);
  }
  sl.ng[idx] = ng;
  sl.row[idx] = row;
  if (FAST) {
    // fp32 gate record: the endpoints as distances along the two source rays. Limits: th * (z + EPS) widened by
    // 0.5% plus 1e-5 of the larger distance (fp32 rounding of the two lambdas and of their difference is below
    // 2e-7 of it, |X_i - X_j| and |lambda_i - lambda_j| agree to 1e-15); see DESIGN.md "gates"
    const double rad = fmax(fabs(c.lam_s), fabs(c.lam_e));
    const double ls = p.l3d.th_scaleinv * (c.zs + consts<double>::eps()) * 1.005 + 1e-5 * rad;
    const double le = p.l3d.th_scaleinv * (c.ze + consts<double>::eps()) * 1.005 + 1e-5 * rad;
    GateRecF g;
    g.dx = (float)d.x; g.dy = (float)d.y; g.dz = (float)d.z; g.lam_e = (float)c.lam_e;
    g.lam_s = (float)c.lam_s; g.lim_s = (float)(ls * 1.000001); g.lim_e = (float)(le * 1.000001);
    g.img = (int)(ng >> 16);
    sl.gatef[idx] = g;
    reinterpret_cast<float *>(sl.psc)[idx] = g.lam_s; // unsorted keys of the depth sort (scratch: the score lists)
  } else {
    // fp32 gate copy, relative to the source camera centre (keeps |coord| ~ depth)
    const vec3<double> rs = c.s - C1, re = c.e - C1;
    // scale-invariance limit th * (z + EPS) widened by 0.5% plus 1e-5 of the coordinate magnitude
    // (fp32 rounding of the two endpoints is < 1e-6 of it); see DESIGN.md "gates"
    const double rad = sqrt(fmax(dot(rs, rs), dot(re, re)));
    const double ls = p.l3d.th_scaleinv * (c.zs + consts<double>::eps()) * 1.005 + 1e-5 * rad;
    const double le = p.l3d.th_scaleinv * (c.ze + consts<double>::eps()) * 1.005 + 1e-5 * rad;
    GateRec g;
    g.dx = (float)d.x; g.dy = (float)d.y; g.dz = (float)d.z; g.lims2 = (float)(ls * ls * 1.000001);
    g.sx = (float)rs.x; g.sy = (float)rs.y; g.sz = (float)rs.z; g.lime2 = (float)(le * le * 1.000001);
    g.ex = (float)re.x; g.ey = (float)re.y; g.ez = (float)re.z;
    g.pad = 0.f;
    sl.gate[idx] = g;
  }
}

// Candidate records of the split path: field-major, field f of slot q at cand[f * cand_stride + q] with q = (row -
// row_begin) * NS + k. Fields (kCandFields in tri_kernels.cuh): sx sy sz ex ey ez zs ze unc lam_s lam_e.
// zs / ze / unc (fields 6..8) of staged candidate i: from shared memory (fused) or from its record (split)
template <bool SPLIT>
LM_D double cand_field(const TriParams &p, const Slab &sl, const double *smem_field, int f, int i, int64_t slot0) {
  if constexpr (SPLIT) return p.cand[f * p.cand_stride + slot0 + sl.row[i]];
  else return smem_field[i];
}

// Phase B of the fast path: all-pairs scoring of the C staged candidates of a node into sl.score.
template <bool SPLIT>
LM_D void phase_b_fast(const TriParams &p, const Slab &sl, const int C, unsigned long long &n1_total,
                       unsigned long long &n2_total) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const unsigned FULL = 0xffffffffu;
  {
    float *ltmp = reinterpret_cast<float *>(sl.psc);
    const int C4 = (C + 3) & ~3;
    if (tid < C4 - C) ltmp[C + tid] = __int_as_float(0x7f800000); // +inf pads: never below a key, never tie-winners
    __syncthreads();
    for (int i = tid; i < C; i += kThreads) {
      const float li = ltmp[i];
      int r = 0;
      for (int j4 = 0; j4 < C4; j4 += 4) {
        const float4 v = *reinterpret_cast<const float4 *>(ltmp + j4);
        r += (v.x < li) || (v.x == li && j4 < i);
        r += (v.y < li) || (v.y == li && j4 + 1 < i);
        r += (v.z < li) || (v.z == li && j4 + 2 < i);
        r += (v.w < li) || (v.w == li && j4 + 3 < i);
      }
      sl.slam[r] = li;
      sl.sidx[r] = (uint16_t)i;
    }
    __syncthreads(); // ltmp (= the score lists) is dead from here on
  }
  const float *slam = sl.slam;
  const uint16_t *sidx = sl.sidx;
  double *psc = sl.psc + (size_t)warp * p.cap;
  uint16_t *pent = sl.pent + (size_t)warp * p.cap;
  // rows are dealt to the warps in equal shares (C = 100: 25 rows per warp, not 32 + 32 + 32 + 4), so the warps
  // reach the barrier before phase C together
  const int n_pass = (C + 32 * kWarps - 1) / (32 * kWarps);
  const int G = (C + kWarps * n_pass - 1) / (kWarps * n_pass); // rows per warp and pass, <= 32
  for (int pass = 0; pass < n_pass; ++pass) {
    const int g0 = (pass * kWarps + warp) * G;
    if (g0 >= C) break;
    const int Gact = min(G, C - g0);
    // B-window, lane = row: two binary searches over the sorted start distances
    int lo = 0, W = 0;
    if (lane < Gact) {
      const float4 a1 = *reinterpret_cast<const float4 *>(&sl.gatef[g0 + lane].lam_s);
      int hi = C;
      if (a1.y < 3e37f) { // (false for inf / NaN limits: the whole node is the window then)
        const float wa = a1.x - a1.y, wb = a1.x + a1.y;
        int l = 0, h = C;
        while (l < h) { const int m = (l + h) >> 1; if (slam[m] < wa) l = m + 1; else h = m; }
        lo = l;
        h = C;
        while (l < h) { const int m = (l + h) >> 1; if (!(slam[m] > wb)) l = m + 1; else h = m; }
        hi = l;
      }
      W = hi - lo;
    }
    int rr = 0;
    while (rr < Gact) {
      // B-gate, one row at a time, lane = window position: the other fp32 gates (end-point interval, angle, other
      // image). The partners of a row are written in ascending candidate order (= ascending neighbour image:
      // candidates are generated image by image) at the running fill of the warp's pair list; lane r keeps the
      // offset and the count of row r of the chunk. A chunk ends when the next row would not fit the list.
      const int cb = rr;
      int fill = 0, off = 0, n = 0;
      for (; rr < Gact; ++rr) {
        const int lo_r = __shfl_sync(FULL, lo, rr), W_r = __shfl_sync(FULL, W, rr);
        const float4 a0 = *reinterpret_cast<const float4 *>(&sl.gatef[g0 + rr].dx);
        const float4 a1 = *reinterpret_cast<const float4 *>(&sl.gatef[g0 + rr].lam_s);
        int n_r = 0;
        if (W_r <= 32) {
          int j = 0x7fffffff;
          bool ok = false;
          if (lane < W_r) {
            j = sidx[lo_r + lane];
            const float4 gj = *reinterpret_cast<const float4 *>(&sl.gatef[j].dx);
            const int imgj = sl.gatef[j].img;
            ok = (imgj != __float_as_int(a1.w)) && !(fabsf(gj.w - a0.w) > a1.z) &&
                 !(fabsf(a0.x * gj.x + a0.y * gj.y + a0.z * gj.z) < p.cos_th3d_f);
          }
          unsigned m = __ballot_sync(FULL, ok);
          n_r = __popc(m);
          if (n_r) {
            if (fill + n_r > p.cap) break; // (a row has fewer than C <= cap partners: an empty list always takes it)
            int rank = 0;
            while (m) { // rank among the partners by candidate index: n_r independent shuffles
              const int t = __ffs((int)m) - 1;
              m &= m - 1;
              rank += __shfl_sync(FULL, j, t) < j;
            }
            if (ok) pent[fill + rank] = (uint16_t)j;
          }
        } else {
          // wide window: partners appended unordered to scratch (the score slots of this chunk's tail are free until
          // B-score), then placed by rank
          uint16_t *tmp = reinterpret_cast<uint16_t *>(psc + fill);
          bool fits = true;
          for (int tb = 0; tb < W_r; tb += 32) {
            const int t = tb + lane;
            int j = 0;
            bool ok = false;
            if (t < W_r) {
              j = sidx[lo_r + t];
              const float4 gj = *reinterpret_cast<const float4 *>(&sl.gatef[j].dx);
              const int imgj = sl.gatef[j].img;
              ok = (imgj != __float_as_int(a1.w)) && !(fabsf(gj.w - a0.w) > a1.z) &&
                   !(fabsf(a0.x * gj.x + a0.y * gj.y + a0.z * gj.z) < p.cos_th3d_f);
            }
            const unsigned m = __ballot_sync(FULL, ok);
            if (fill + n_r + __popc(m) > p.cap) { fits = false; break; }
            if (ok) tmp[n_r + __popc(m & lt_mask)] = (uint16_t)j;
            n_r += __popc(m);
          }
          if (!fits) break;
          __syncwarp();
          // (tmp occupies 2 bytes per partner inside psc[fill ..), pent[fill ..) is a different array)
          for (int e = lane; e < n_r; e += 32) {
            const uint16_t v = tmp[e];
            int rank = 0;
            for (int x = 0; x < n_r; ++x) rank += tmp[x] < v;
            pent[fill + rank] = v;
          }
        }
        if (lane == rr) { off = fill; n = n_r; }
        fill += n_r;
      }
      const int ce = rr;
      n1_total += (unsigned long long)fill;
      __syncwarp();
      // B-score: exact reference scores, lane = pair
      for (int fb = 0; fb < fill; fb += 32) {
        const int f = fb + lane;
        int r = cb; // largest row of the chunk whose offset is <= f (rows without partners share the next offset)
#pragma unroll
        for (int step = 16; step >= 1; step >>= 1) {
          const int cand = r + step;
          const int v = __shfl_sync(FULL, off, cand & 31);
          if (cand < ce && v <= f) r = cand;
        }
        if (f < fill) {
          const int j = pent[f];
          psc[f] = pair_score_fast<SPLIT>(p, sl, g0 + r, j, (uint32_t)sl.gatef[j].img);
        }
      }
      n2_total += (unsigned long long)fill;
      __syncwarp();
      // B-sum: one image contributes its maximum once (:110-112), images in ascending order (the partners of a row
      // are sorted by candidate index, i.e. by image)
      if (lane >= cb && lane < ce) {
        double sum = 0.0, mx = 0.0;
        int cur = -1;
        for (int e = 0; e < n; ++e) {
          const int im = sl.gatef[pent[off + e]].img;
          const double sc = psc[off + e];
          if (im != cur) { sum += mx; cur = im; mx = sc; }
          else mx = (mx > sc) ? mx : sc;
        }
        sum += mx;
        sl.score[g0 + lane] = sum;
      }
      __syncwarp();
    }
  }
}

// Phase C: valid connections + best candidate (:115-153) of the node whose rows start at r0. slot0 is the record slot
// of the node's first row (split path only).
template <int NS, bool SPLIT>
LM_D void phase_c(const TriParams &p, const Slab &sl, const int C, const uint32_t r0, NodeRecord *rec, int &s_nvalid,
                  int64_t slot0 = 0) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int nvalid_local = 0;
  for (int i = tid; i < C; i += kThreads) {
    const double sc = sl.score[i];
    bool valid = sc >= p.fullscore_th; // `if (score < fullscore_th) continue;`
    if (valid && C > p.max_valid_conns) {
      // rank in the (score, tri_id) descending order of std::greater<pair<double,int>> (:128-129)
      int rank = 0;
      for (int k = 0; k < C; ++k) {
        const double sk = sl.score[k];
        rank += (sk > sc) || (sk == sc && k > i);
      }
      valid = rank < p.max_valid_conns;
    }
    p.row_state[(int64_t)r0 * NS + sl.row[i]] = valid ? 2 : 1;
    nvalid_local += valid;
    if (p.row_cand) {
      double *o = p.row_cand + ((int64_t)r0 * NS + sl.row[i]) * 10;
      o[0] = sl.sx[i]; o[1] = sl.sy[i]; o[2] = sl.sz[i]; o[3] = sl.ex[i]; o[4] = sl.ey[i]; o[5] = sl.ez[i];
      o[6] = cand_field<SPLIT>(p, sl, sl.zs, 6, i, slot0); o[7] = cand_field<SPLIT>(p, sl, sl.ze, 7, i, slot0);
      o[8] = cand_field<SPLIT>(p, sl, sl.unc, 8, i, slot0); o[9] = sc;
    }
  }
  if (nvalid_local) atomicAdd(&s_nvalid, nvalid_local);
  // best: first strict maximum from max_score = -1 (:145-153) == max score, lowest index on ties.
  if (warp == 0) {
    double bs = -1.0;
    int bi = -1;
    for (int i = lane; i < C; i += 32) {
      const double sc = sl.score[i];
      if (sc > bs) { bs = sc; bi = i; }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const double os = __shfl_down_sync(0xffffffffu, bs, d);
      const int oi = __shfl_down_sync(0xffffffffu, bi, d);
      if (oi >= 0 && (os > bs || (os == bs && (bi < 0 || oi < bi)))) { bs = os; bi = oi; }
    }
    bi = __shfl_sync(0xffffffffu, bi, 0);
    if (bi >= 0) {
      if (lane < 3) rec->line[lane] = (lane == 0) ? sl.sx[bi] : (lane == 1 ? sl.sy[bi] : sl.sz[bi]);
      else if (lane < 6) rec->line[lane] = (lane == 3) ? sl.ex[bi] : (lane == 4 ? sl.ey[bi] : sl.ez[bi]);
      else if (lane == 6) rec->line[6] = cand_field<SPLIT>(p, sl, sl.zs, 6, bi, slot0);
      else if (lane == 7) rec->line[7] = cand_field<SPLIT>(p, sl, sl.ze, 7, bi, slot0);
      else if (lane == 8) rec->line[8] = cand_field<SPLIT>(p, sl, sl.unc, 8, bi, slot0);
      else if (lane == 9) rec->score = sl.score[bi];
      else if (lane == 10) { rec->ng_view = (int32_t)(sl.ng[bi] >> 16); rec->ng_line = (int32_t)(sl.ng[bi] & 0xffffu); }
    } else {
      if (lane < 9) rec->line[lane] = (lane == 8) ? -1.0 : 0.0;
      if (lane == 9) rec->score = 0.0;
      if (lane == 10) { rec->ng_view = 0; rec->ng_line = 0; }
    }
  }
}

// FAST: reduced-form scorer and plane-pair triangulation only (the default configuration); the generic
// instantiation keeps the reference-structured scorer, the 2d margin gates and endpoint triangulation. Splitting
// them keeps the hot kernel's code (and instruction-cache footprint) small.
template <bool SLAB, bool VP, bool FAST>
__global__ void __launch_bounds__(kThreads, LM_TRI_MIN_BLOCKS) tri_node_kernel(const __grid_constant__ TriParams p) {
  constexpr int NS = VP ? 3 : 1; // proposal slots per match row: [vp1, vp2, algebraic] (base_line_triangulator.cc:258-326)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_wtot[kWarps];
  __shared__ int s_nvalid;
  __shared__ int s_next_row;
  __shared__ __align__(8) unsigned long long s_mbar; // completion of the neighbour-view bulk copies of a node
  uint32_t mbar_parity = 0;
  if constexpr (FAST && !SLAB && (LM_TRI_TMA || VP)) {
    if (threadIdx.x == 0) mbar_init(&s_mbar, 1);
    __syncthreads();
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  Slab sl;
  if (SLAB) sl.carve(p.slab + (int64_t)blockIdx.x * p.slab_stride, p.cap, FAST);
  else sl.carve(reinterpret_cast<char *>(smem_raw), p.cap, FAST);
  uint32_t *list1 = FAST ? nullptr : sl.list + (size_t)(warp * 2) * (p.cap + kListExtra);
  uint32_t *list2 = FAST ? nullptr : list1 + p.cap + kListExtra;
  uint16_t *list0 = FAST ? nullptr : sl.list0 + (size_t)warp * p.cap;
  unsigned long long n1_total = 0, n2_total = 0;

  for (int64_t node = p.node_begin + blockIdx.x; node < p.node_end; node += gridDim.x) {
    const uint32_t r0 = p.node_row_off[node], r1 = p.node_row_off[node + 1];
    const int nrows = (int)(r1 - r0);
    NodeRecord *rec = &p.nodes[node];
    if (nrows == 0 || nrows * NS > p.cap) {
      if (tid < 9) rec->line[tid] = (tid == 8) ? -1.0 : 0.0;
      if (tid == 9) { rec->score = 0.0; rec->ng_view = 0; rec->ng_line = 0; rec->n_cand = 0; rec->n_valid = 0; }
      if (nrows != 0 && tid == 10) *p.overflow = 1; // staging area sized from a stale hint: the host repeats the run
      continue;
    }
    // ---------------- phase A: candidate generation with stable compaction -----------------
    // ---- neighbour views of the node -> shared memory. Rows are ordered by neighbour view, so a new view starts where
    // the view index changes; the thread that sees the change issues one 208-byte TMA bulk copy (cp.async.bulk,
    // completion on an mbarrier) into the view's slot. Phase A then reads K|R|t-derived blocks from shared memory
    // instead of chasing row -> view index -> global view record. The staging area aliases the phase-B score lists.
    const ViewD *sviews = nullptr;
    const uint8_t *slot_of_row = nullptr;
    int n_stage = 0;
    if constexpr (FAST && !SLAB && (LM_TRI_TMA || VP)) {
      const int stage_off = p.cap * 4; // the depth-sort keys written by phase A come first
      ViewD *sv = reinterpret_cast<ViewD *>(reinterpret_cast<char *>(sl.psc) + stage_off);
      uint8_t *slots = reinterpret_cast<uint8_t *>(sl.sidx); // [nrows <= cap]; rewritten by the depth sort afterwards
      const int stage_cap = min(255, (int)(((size_t)kWarps * p.cap * 8 - stage_off) / sizeof(ViewD)));
      int carry = 0;
      for (int base = 0; base < nrows; base += kThreads) {
        const int r = base + tid;
        uint32_t view = 0;
        int flag = 0;
        if (r < nrows) {
          view = __ldg(&p.row_ng[r0 + r]) >> 16;
          flag = (r == 0) || ((__ldg(&p.row_ng[r0 + r - 1]) >> 16) != view);
        }
        int incl = flag;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int o = __shfl_up_sync(0xffffffffu, incl, d);
          if (lane >= d) incl += o;
        }
        if (lane == 31) s_wtot[warp] = incl;
        __syncthreads();
        int woff = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
          if (w < warp) woff += s_wtot[w];
          tot += s_wtot[w];
        }
        const int slot = carry + woff + incl - 1;
        if (r < nrows) slots[r] = (uint8_t)min(slot, 255);
        if (flag && slot < stage_cap) bulk_copy_g2s(sv + slot, p.views + view, (uint32_t)sizeof(ViewD), &s_mbar);
        carry += tot;
        __syncthreads();
      }
      n_stage = min(carry, stage_cap);
      if (tid == 0) mbar_arrive_expect_tx(&s_mbar, (uint32_t)(n_stage * sizeof(ViewD)));
      sviews = sv;
      slot_of_row = slots; // (the copies are awaited after the source-line constants below: their latency is hidden)
    }
    const uint32_t v1i = p.node_view[node];
    const ViewD &v1 = p.views[v1i];
    Src src;
    src.l1 = ld_seg(&p.segs[node]);
    {
      double dx = src.l1.x - src.l1.z, dy = src.l1.y - src.l1.w;
      src.ok = !(sqrt(dx * dx + dy * dy) <= p.min_length_2d); // :166
      src.w1s = mat3_mul_h(v1.M, src.l1.x, src.l1.y);
      src.w1e = mat3_mul_h(v1.M, src.l1.z, src.l1.w);
      src.ray1s = normalized(src.w1s);
      src.ray1e = normalized(src.w1e);
      src.C1 = mk3(v1.C[0], v1.C[1], v1.C[2]);
      src.n1 = normalized(cross(src.w1s, src.w1e));
    }
    if constexpr (FAST && !SLAB && (LM_TRI_TMA || VP)) {
      mbar_wait(&s_mbar, mbar_parity);
      mbar_parity ^= 1u;
    }
    int count = 0;
    for (int base = 0; base < nrows; base += kThreads) {
      const int r = base + tid;
      Cand cs[NS];
      bool oks[NS];
#pragma unroll
      for (int k = 0; k < NS; ++k) oks[k] = false;
      double4 l2 = make_double4(0, 0, 0, 0);
      uint32_t ng = 0;
      if (r < nrows && src.ok) {
        ng = __ldg(&p.row_ng[r0 + r]);
        const uint32_t ngv = ng >> 16, ngl = ng & 0xffffu;
        if (VP) {
          // Step 2 (:258-288): proposals from the VP of the source line and of the matched line; both use view 1
          const double4 l2v = ld_seg(&p.segs[p.line_off[ngv] + ngl]);
          const double ddx = l2v.x - l2v.z, ddy = l2v.y - l2v.w;
          if (!(sqrt(ddx * ddx + ddy * ddy) <= p.min_length_2d) && !p.disable_vp) {
            const ViewD *v2q = &p.views[ngv];
            if constexpr (FAST && !SLAB && (LM_TRI_TMA || VP)) {
              const int slot = slot_of_row[r];
              if (slot < n_stage) v2q = &sviews[slot];
            }
            const ViewD &v2 = *v2q;
            const vec3<double> c2s = mat3_mul_h(v2.M, l2v.x, l2v.y), c2e = mat3_mul_h(v2.M, l2v.z, l2v.w);
            const int lab1 = p.vp_label[node];
            if (lab1 >= 0) {
              const double *vp = p.vps + 3 * (p.vp_off[v1i] + lab1);
              oks[0] = gen_vp_candidate(p, v1, v2, src, c2s, c2e, normalized(mat3_mul(v1.M, mk3(vp[0], vp[1], vp[2]))), cs[0]);
            }
            const int lab2 = p.vp_label[p.line_off[ngv] + ngl];
            if (lab2 >= 0) {
              const double *vp = p.vps + 3 * (p.vp_off[ngv] + lab2);
              oks[1] = gen_vp_candidate(p, v1, v2, src, c2s, c2e, normalized(mat3_mul(v1.M, mk3(vp[0], vp[1], vp[2]))), cs[1]);
            }
          }
          l2 = l2v;
        }
        const ViewD *v2p = &p.views[ngv];
        if constexpr (FAST && !SLAB && (LM_TRI_TMA || VP)) {
          const int slot = slot_of_row[r];
          if (slot < n_stage) v2p = &sviews[slot];
        }
        oks[NS - 1] = gen_candidate<!FAST>(p, v1, *v2p, src, ngv, ngl, cs[NS - 1], l2);
      }
      int cnt = 0;
#pragma unroll
      for (int k = 0; k < NS; ++k) {
        if (r < nrows) p.row_state[(int64_t)(r0 + r) * NS + k] = 0;
        cnt += oks[k];
      }
      // stable compaction: exclusive prefix of the per-row candidate counts
      int incl = cnt;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
      }
      if (lane == 31) s_wtot[warp] = incl;
      __syncthreads();
      int woff = 0, tot = 0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) {
        if (w < warp) woff += s_wtot[w];
        tot += s_wtot[w];
      }
      int idx = count + woff + incl - cnt;
#pragma unroll
      for (int k = 0; k < NS; ++k) {
        if (!oks[k]) continue;
        stage_cand<FAST, false>(p, sl, idx, cs[k], l2, ng, (uint32_t)r * NS + k, src.C1);
        ++idx;
      }
      count += tot;
      __syncthreads();
    }
    const int C = count;
    if (tid == 0) { s_nvalid = 0; s_next_row = 0; }
    __syncthreads();
    // ---------------- phase B: all-pairs scoring ------------------------------------------------
    if constexpr (FAST) {
      // All candidates of the node start on one ray and end on another (GateRecF), so "l_j can score against l_i"
      // needs |lam_s(j) - lam_s(i)| <= lim_s(i): after a sort by lam_s the partners of a row are a contiguous window.
      //   B-sort   rank sort of the candidates by lam_s (ties by index), whole CTA
      //   per warp, 32 rows at a time (lane = row):
      //   B-window two binary searches per row
      //   B-gate   the other fp32 gates (end-point interval, angle, other image) over the window, twice: count, then
      //            write -- each row's partners land contiguously in the warp's pair list, no atomics, no compaction
      //   B-score  exact fp64 scores of the pair list, 32 pairs per step (lane = pair; rows found by a search over
      //            the lanes' offsets)
      //   B-sum    lane = row again: maximum per neighbour image, images added in ascending order -- the order of the
      //            reference's std::map (:105-112), so a row's total does not depend on how the work was split.
      // Pruned pairs would have scored exactly 0 (DESIGN.md "Exactness argument"); every surviving pair is scored by
      // pair_score_fast in fp64.
      phase_b_fast<false>(p, sl, C, n1_total, n2_total);
      __syncthreads();
    } else {
    // Warps fetch rows i dynamically. B1 prunes (i, j) pairs with the fp32 3d gates and appends the
    // survivors of several rows to a warp-private list until it holds >= kFlush entries, so that the fp64
    // stages B2 (2d margin gates) and B3 (exact reference score) run on dense 32-lane batches.
    for (int i = tid; i < C; i += kThreads) sl.score[i] = 0.0;
    // records up to the next multiple of 32 can never pass the start-point test: the prefilter loop needs no bounds
    if (tid < 32 && C + tid < ((C + 31) & ~31)) {
      GateRec z;
      z.dx = z.dy = z.dz = 0.f; z.lims2 = 0.f;
      z.sx = z.sy = z.sz = 3e18f; z.lime2 = 0.f;
      z.ex = z.ey = z.ez = 3e18f; z.pad = 0.f;
      sl.gate[C + tid] = z;
    }
    __syncthreads();
    bool more = true;
    while (more) {
      int n1 = 0;
      while (n1 < kFlush) {
        int i = 0;
        if (lane == 0) i = atomicAdd(&s_next_row, 1);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= C) { more = false; break; }
        const GateRec rf = sl.gate[i];
        const uint32_t vi = sl.ng[i] >> 16;
        // B0: start-point prefilter. The scale-invariant endpoint test (line_linker.cc:269-277, th_scaleinv of the
        // depth) is by far the most selective 3d test, so its start-point half runs first on every candidate (one
        // 16-byte load, 8 flops); the other gates only see the survivors. (A byte-hash of the log distance tested
        // four candidates per lane was measured slower: more false positives reach B1 than it saves here.)
        int n0 = 0;
        for (int jb = 0; jb < C; jb += 32) {
          const int j = jb + lane;
          const float4 b = *reinterpret_cast<const float4 *>(&sl.gate[j].sx);
          const float ax = rf.sx - b.x, ay = rf.sy - b.y, az = rf.sz - b.z;
          const bool pass = !(ax * ax + ay * ay + az * az > rf.lims2);
          const unsigned bal = __ballot_sync(0xffffffffu, pass);
          if (pass) list0[n0 + __popc(bal & lt_mask)] = (uint16_t)j;
          n0 += __popc(bal);
        }
        __syncwarp();
        // B1: the other fp32 3d gates (angle, end point) and the same-image exclusion (which also drops j == i)
        for (int kb = 0; kb < n0; kb += 32) {
          const int k = kb + lane;
          bool pass = false;
          int j = 0;
          if (k < n0) {
            j = list0[k];
            pass = (sl.ng[j] >> 16) != vi && gate3d_rest(rf, &sl.gate[j], p.cos_th3d_f);
          }
          const unsigned bal = __ballot_sync(0xffffffffu, pass);
          if (pass) list1[n1 + __popc(bal & lt_mask)] = ((uint32_t)i << 16) | (uint32_t)j;
          n1 += __popc(bal);
        }
        __syncwarp();
      }
      __syncwarp();
      n1_total += n1;
      if (n1 == 0) continue;
      // B2 (only with the reference-structured scorer): fp64 margin gates of the 2d tests
      int n2 = n1;
      uint32_t *listS = list1;
      if (!FAST) {
        n2 = 0;
        for (int kb = 0; kb < n1; kb += 32) {
          const int k = kb + lane;
          bool pass = false;
          uint32_t e = 0;
          if (k < n1) {
            e = list1[k];
            const int i = e >> 16, j = e & 0xffffu;
            seg<vec3<double>> Li;
            Li.s = mk3(sl.sx[i], sl.sy[i], sl.sz[i]);
            Li.e = mk3(sl.ex[i], sl.ey[i], sl.ez[i]);
            pass = gate2d(p, Li, sl, j, sl.ng[j] >> 16);
          }
          const unsigned bal = __ballot_sync(0xffffffffu, pass);
          if (pass) list2[n2 + __popc(bal & lt_mask)] = e;
          n2 += __popc(bal);
        }
        __syncwarp();
        listS = list2;
      }
      n2_total += n2;
      // B3: exact reference scores; maximum per (row, image), summed per row (:97-112). Entries are ordered
      // by (row, image), so both reductions are segmented warp scans with a carry across batches.
      uint32_t carry_key = 0xffffffffu, cur_row = 0xffffffffu;
      double carry_max = 0.0, cur_sum = 0.0;
      for (int kb = 0; kb < n2; kb += 32) {
        const int k = kb + lane;
        double sc = 0.0;
        uint32_t key = 0xfffffffeu, row = 0xfffffffeu; // key = row << 16 | view
        if (k < n2) {
          const uint32_t e = listS[k];
          const int i = e >> 16, j = e & 0xffffu;
          const uint32_t vj = sl.ng[j] >> 16;
          row = (uint32_t)i;
          key = (row << 16) | vj;
          if (FAST) sc = pair_score_fast(p, sl, i, j, vj);
          else {
            seg<vec3<double>> Li;
            Li.s = mk3(sl.sx[i], sl.sy[i], sl.sz[i]);
            Li.e = mk3(sl.ex[i], sl.ey[i], sl.ez[i]);
            sc = pair_score(p, Li, mk3(sl.dx[i], sl.dy[i], sl.dz[i]), sl.zs[i], sl.ze[i], sl, j, vj);
          }
        }
        if (key == carry_key && carry_max > sc) sc = carry_max;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const double o = __shfl_up_sync(0xffffffffu, sc, d);
          const uint32_t ok = __shfl_up_sync(0xffffffffu, key, d);
          if (lane >= d && ok == key && o > sc) sc = o;
        }
        uint32_t knext = __shfl_down_sync(0xffffffffu, key, 1);
        if (lane == 31) {
          knext = 0xfffffffdu;
          if (k + 1 < n2) { const uint32_t e2 = listS[k + 1]; knext = (e2 & 0xffff0000u) | (sl.ng[e2 & 0xffffu] >> 16); }
        }
        const bool seg_end = (k < n2) && (knext != key);
        // one image contributes its maximum once (:110-112): add the segment maxima to their row's total in
        // list order = ascending (row, image), exactly the reference's std::map order; the running
        // (row, sum) pair is warp-uniform, so the result does not depend on how rows were batched
        unsigned m = __ballot_sync(0xffffffffu, seg_end);
        while (m) {
          const int l = __ffs(m) - 1;
          const double v = __shfl_sync(0xffffffffu, sc, l);
          const uint32_t r = __shfl_sync(0xffffffffu, row, l);
          if (r != cur_row) {
            if (cur_row != 0xffffffffu && lane == 0) sl.score[cur_row] = cur_sum;
            cur_row = r;
            cur_sum = 0.0;
          }
          cur_sum += v;
          m &= m - 1;
        }
        const uint32_t k31 = __shfl_sync(0xffffffffu, key, 31);
        const double s31 = __shfl_sync(0xffffffffu, sc, 31);
        const bool end31 = __shfl_sync(0xffffffffu, (int)seg_end, 31);
        if (!end31 && kb + 31 < n2) { carry_key = k31; carry_max = s31; }
        else { carry_key = 0xffffffffu; carry_max = 0.0; }
      }
      if (cur_row != 0xffffffffu && lane == 0) sl.score[cur_row] = cur_sum;
      __syncwarp();
    }
    __syncthreads();
    } // generic phase B
    // ---------------- phase C: valid connections + best candidate (:115-153) ----------------
    phase_c<NS, false>(p, sl, C, r0, rec, s_nvalid);
    __syncthreads();
    if (tid == 0) {
      rec->n_cand = C;
      rec->n_valid = s_nvalid;
      if (C) atomicAdd(&p.counters[0], (unsigned long long)C);
      if (s_nvalid) atomicAdd(&p.counters[1], (unsigned long long)s_nvalid);
    }
    __syncthreads();
  }
  if (lane == 0 && n1_total) {
    atomicAdd(&p.counters[2], n1_total); // pairs past the fp32 3d gates
    atomicAdd(&p.counters[3], n2_total); // pairs scored exactly in fp64
  }
}

template <bool VP, bool FAST> static cudaError_t launch_tri_vf(const TriParams &p, int grid, size_t smem, cudaStream_t s) {
  if (p.use_slab) {
    tri_node_kernel<true, VP, FAST><<<grid, kThreads, 0, s>>>(p);
    return cudaGetLastError();
  }
  // the opt-in is per device (and per function): set it on every launch above the default limit
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(tri_node_kernel<false, VP, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  tri_node_kernel<false, VP, FAST><<<grid, kThreads, smem, s>>>(p);
  return cudaGetLastError();
}
cudaError_t launch_tri_node_kernel(const TriParams &p, int grid, int block, size_t smem, cudaStream_t s) {
  (void)block;
  const bool fast = p.fast_forms && !p.use_endpoints_triangulation;
  if (p.use_vp) return fast ? launch_tri_vf<true, true>(p, grid, smem, s) : launch_tri_vf<true, false>(p, grid, smem, s);
  return fast ? launch_tri_vf<false, true>(p, grid, smem, s) : launch_tri_vf<false, false>(p, grid, smem, s);
}

// ---- split fast path ------------------------------------------------------------------------------------------------
// The fused kernel holds phase A's fp64 registers and the scorer's staging area in one CTA, which caps it at 4 CTAs/SM.
// Split, each part runs at its own occupancy: generation is flat (one thread per match row, no shared memory, no
// barriers) and writes each candidate as a record to global memory; scoring is one CTA per node sized from the real
// candidate count. The same fp64 values cross the boundary and the same expressions run on them, so the results are
// those of the fused kernel.
#ifndef LM_GEN_THREADS
#define LM_GEN_THREADS 128
#endif
#ifndef LM_SCORE_MIN_BLOCKS
#define LM_SCORE_MIN_BLOCKS 6
#endif

// One thread per match row of the group: phase A of tri_node_kernel without the compaction. Writes row_state = 0 / 1
// for every proposal slot and the record of every candidate.
template <bool VP>
__global__ void __launch_bounds__(LM_GEN_THREADS, VP ? 2 : 3) tri_gen_kernel(const __grid_constant__ TriParams p) {
  constexpr int NS = VP ? 3 : 1;
  const int64_t r = p.row_begin + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= p.row_end) return;
  const uint32_t node = __ldg(&p.row_node[r]);
  const uint32_t v1i = p.node_view[node];
  const ViewD &v1 = p.views[v1i];
  Src src;
  src.l1 = ld_seg(&p.segs[node]);
  {
    double dx = src.l1.x - src.l1.z, dy = src.l1.y - src.l1.w;
    src.ok = !(sqrt(dx * dx + dy * dy) <= p.min_length_2d); // :166
    src.w1s = mat3_mul_h(v1.M, src.l1.x, src.l1.y);
    src.w1e = mat3_mul_h(v1.M, src.l1.z, src.l1.w);
    src.ray1s = normalized(src.w1s);
    src.ray1e = normalized(src.w1e);
    src.C1 = mk3(v1.C[0], v1.C[1], v1.C[2]);
    src.n1 = normalized(cross(src.w1s, src.w1e));
  }
  Cand cs[NS];
  bool oks[NS];
#pragma unroll
  for (int k = 0; k < NS; ++k) oks[k] = false;
  if (src.ok) {
    const uint32_t ng = __ldg(&p.row_ng[r]);
    const uint32_t ngv = ng >> 16, ngl = ng & 0xffffu;
    const ViewD &v2 = p.views[ngv];
    double4 l2;
    if (VP) {
      // Step 2 (:258-288): proposals from the VP of the source line and of the matched line; both use view 1
      const double4 l2v = ld_seg(&p.segs[p.line_off[ngv] + ngl]);
      const double ddx = l2v.x - l2v.z, ddy = l2v.y - l2v.w;
      if (!(sqrt(ddx * ddx + ddy * ddy) <= p.min_length_2d) && !p.disable_vp) {
        const vec3<double> c2s = mat3_mul_h(v2.M, l2v.x, l2v.y), c2e = mat3_mul_h(v2.M, l2v.z, l2v.w);
        const int lab1 = p.vp_label[node];
        if (lab1 >= 0) {
          const double *vp = p.vps + 3 * (p.vp_off[v1i] + lab1);
          oks[0] = gen_vp_candidate(p, v1, v2, src, c2s, c2e, normalized(mat3_mul(v1.M, mk3(vp[0], vp[1], vp[2]))), cs[0]);
        }
        const int lab2 = p.vp_label[p.line_off[ngv] + ngl];
        if (lab2 >= 0) {
          const double *vp = p.vps + 3 * (p.vp_off[ngv] + lab2);
          oks[1] = gen_vp_candidate(p, v1, v2, src, c2s, c2e, normalized(mat3_mul(v1.M, mk3(vp[0], vp[1], vp[2]))), cs[1]);
        }
      }
    }
    oks[NS - 1] = gen_candidate<false>(p, v1, v2, src, ngv, ngl, cs[NS - 1], l2);
  }
  const int64_t q0 = (r - p.row_begin) * NS;
#pragma unroll
  for (int k = 0; k < NS; ++k) {
    p.row_state[r * NS + k] = oks[k] ? 1 : 0;
    if (!oks[k]) continue;
    const Cand &c = cs[k];
    double *o = p.cand + q0 + k;
    const int64_t st = p.cand_stride;
    o[0] = c.s.x; o[st] = c.s.y; o[2 * st] = c.s.z; o[3 * st] = c.e.x; o[4 * st] = c.e.y; o[5 * st] = c.e.z;
    o[6 * st] = c.zs; o[7 * st] = c.ze; o[8 * st] = c.unc; o[9 * st] = c.lam_s; o[10 * st] = c.lam_e;
  }
}

// One CTA per node: the node's candidate slots (row_state == 1) in slot order -- the order of the fused kernel's stable
// compaction, so candidate indices are the same -- staged from their records, then phases B and C of the fused kernel.
template <bool VP>
__global__ void __launch_bounds__(kThreads, LM_SCORE_MIN_BLOCKS) tri_score_kernel(const __grid_constant__ TriParams p) {
  constexpr int NS = VP ? 3 : 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_wtot[kWarps];
  __shared__ int s_nvalid;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  Slab sl;
  sl.carve_split(reinterpret_cast<char *>(smem_raw), p.cap);
  unsigned long long n1_total = 0, n2_total = 0;
  for (int64_t node = p.node_begin + blockIdx.x; node < p.node_end; node += gridDim.x) {
    const uint32_t r0 = p.node_row_off[node], r1 = p.node_row_off[node + 1];
    const int nslots = (int)(r1 - r0) * NS;
    NodeRecord *rec = &p.nodes[node];
    // compaction of the candidate slots
    int count = 0;
    for (int base = 0; base < nslots; base += kThreads) {
      const int q = base + tid;
      const bool cand = q < nslots && p.row_state[(int64_t)r0 * NS + q] == 1;
      const unsigned m = __ballot_sync(0xffffffffu, cand);
      if (lane == 0) s_wtot[warp] = __popc(m);
      __syncthreads();
      int woff = 0, tot = 0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) {
        if (w < warp) woff += s_wtot[w];
        tot += s_wtot[w];
      }
      const int idx = count + woff + __popc(m & lt_mask);
      if (cand && idx < p.cap) sl.row[idx] = (uint32_t)q;
      count += tot;
      __syncthreads();
    }
    const int C = count;
    if (tid == 0 && C) atomicMax(p.max_cand, (unsigned int)C);
    if (C > p.cap) { // staging area sized from a stale hint: the host repeats the run with the exact size
      if (tid < 9) rec->line[tid] = (tid == 8) ? -1.0 : 0.0;
      if (tid == 9) { rec->score = 0.0; rec->ng_view = 0; rec->ng_line = 0; rec->n_cand = 0; rec->n_valid = 0; }
      if (tid == 10) *p.overflow = 1;
      continue;
    }
    // ---- staging from the records (phase A's derivation)
    const int64_t slot0 = (int64_t)(r0 - p.row_begin) * NS;
    for (int i = tid; i < C; i += kThreads) {
      const uint32_t q = sl.row[i];
      const double *o = p.cand + slot0 + q;
      const int64_t st = p.cand_stride;
      Cand c;
      c.s = mk3(o[0], o[st], o[2 * st]);
      c.e = mk3(o[3 * st], o[4 * st], o[5 * st]);
      c.zs = o[6 * st]; c.ze = o[7 * st]; c.unc = o[8 * st]; c.lam_s = o[9 * st]; c.lam_e = o[10 * st];
      const uint32_t ng = __ldg(&p.row_ng[r0 + q / NS]);
      const uint32_t segi = (uint32_t)(p.line_off[ng >> 16] + (ng & 0xffffu));
      stage_cand<true, true>(p, sl, i, c, ld_seg(&p.segs[segi]), ng, q, mk3(0.0, 0.0, 0.0), segi); // (C1: generic layout only)
    }
    if (tid == 0) s_nvalid = 0;
    __syncthreads();
    phase_b_fast<true>(p, sl, C, n1_total, n2_total);
    __syncthreads();
    phase_c<NS, true>(p, sl, C, r0, rec, s_nvalid, slot0);
    __syncthreads();
    if (tid == 0) {
      rec->n_cand = C;
      rec->n_valid = s_nvalid;
      if (C) atomicAdd(&p.counters[0], (unsigned long long)C);
      if (s_nvalid) atomicAdd(&p.counters[1], (unsigned long long)s_nvalid);
    }
    __syncthreads();
  }
  if (lane == 0 && n1_total) {
    atomicAdd(&p.counters[2], n1_total); // pairs past the fp32 3d gates
    atomicAdd(&p.counters[3], n2_total); // pairs scored exactly in fp64
  }
}

template <bool VP> static cudaError_t launch_split_v(const TriParams &p, int grid, size_t smem, cudaStream_t s) {
  const int64_t rows = p.row_end - p.row_begin;
  if (rows > 0) {
    tri_gen_kernel<VP><<<(unsigned)((rows + LM_GEN_THREADS - 1) / LM_GEN_THREADS), LM_GEN_THREADS, 0, s>>>(p);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(tri_score_kernel<VP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  tri_score_kernel<VP><<<grid, kThreads, smem, s>>>(p);
  return cudaGetLastError();
}
cudaError_t launch_tri_split(const TriParams &p, int grid, size_t smem, cudaStream_t s) {
  return p.use_vp ? launch_split_v<true>(p, grid, smem, s) : launch_split_v<false>(p, grid, smem, s);
}

// The per-run block tables (match tables ordered by (source view, neighbour), row offsets) are derived on the
// device from block descriptors that were uploaded together with the matches. Nothing has to cross PCIe when
// a run starts: any host->device transfer issued then (copy-engine copies, large kernel parameters, even
// zero-copy reads) was measured to wait ~3 ms behind a 160 MB match upload still in flight.
__global__ void block_keys_kernel(const RawBlock *__restrict__ raw, int n_all, int vb, int ve, int exhaustive,
                                  uint32_t *__restrict__ key, uint32_t *__restrict__ val) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_all) return;
  const RawBlock b = raw[i];
  const bool in = b.src_view >= vb && b.src_view < ve;
  key[i] = in ? (((uint32_t)b.src_view << 16) | (uint32_t)(exhaustive ? b.order : b.ng_view)) : 0xffffffffu;
  val[i] = (uint32_t)i;
}
__global__ void block_gather_kernel(const RawBlock *__restrict__ raw, const uint32_t *__restrict__ sorted_idx, int nb,
                                    int32_t *__restrict__ blk_src, int32_t *__restrict__ blk_ng,
                                    int64_t *__restrict__ blk_pair_off, int64_t *__restrict__ blk_rows) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > nb) return;
  if (i == nb) { blk_rows[i] = 0; return; }
  const RawBlock b = raw[sorted_idx[i]];
  blk_src[i] = b.src_view;
  blk_ng[i] = b.ng_view;
  blk_pair_off[i] = b.pair_off;
  blk_rows[i] = b.n_rows;
}
void launch_block_keys(const RawBlock *raw, int n_all, int vb, int ve, int exhaustive, uint32_t *key, uint32_t *val,
                       cudaStream_t s) {
  if (n_all <= 0) return;
  block_keys_kernel<<<(n_all + 255) / 256, 256, 0, s>>>(raw, n_all, vb, ve, exhaustive, key, val);
}
void launch_block_gather(const RawBlock *raw, const uint32_t *sorted_idx, int nb, int32_t *blk_src, int32_t *blk_ng,
                         int64_t *blk_pair_off, int64_t *blk_rows, cudaStream_t s) {
  block_gather_kernel<<<(nb + 1 + 255) / 256, 256, 0, s>>>(raw, sorted_idx, nb, blk_src, blk_ng, blk_pair_off, blk_rows);
}
__global__ void zero_words_kernel(unsigned int *p, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0u;
}
// cudaMemsetAsync may be routed to a copy engine and then waits behind a running match upload
void launch_zero_words(void *d_dst, int n_words, cudaStream_t s) {
  zero_words_kernel<<<(n_words + 127) / 128, 128, 0, s>>>(static_cast<unsigned int *>(d_dst), n_words);
}

// ------------------------------------------------------------------------------------------------
// Match tables -> node-major rows. Flat row order = (source view asc, neighbour view asc, row), the
// order in which TriangulateImage appends to tris_ (base_line_triangulator.cc:74-100); a stable sort
// by node id then yields each node's candidates in reference order.
__global__ void expand_rows_kernel(const int32_t *__restrict__ pairs, const int64_t *__restrict__ blk_row_off,
                                   const int32_t *__restrict__ blk_src, const int32_t *__restrict__ blk_ng,
                                   const int64_t *__restrict__ blk_pair_off, int n_blocks,
                                   const int64_t *__restrict__ line_off, int64_t r_begin, int64_t n_rows,
                                   uint32_t *__restrict__ key, uint32_t *__restrict__ val, int *err) {
  for (int64_t r = r_begin + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n_rows;
       r += (int64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = n_blocks; // largest b with blk_row_off[b] <= r
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (blk_row_off[mid] <= r) lo = mid; else hi = mid;
    }
    const int b = lo;
    const int64_t q = blk_pair_off[b] + (r - blk_row_off[b]);
    const int2 pr = reinterpret_cast<const int2 *>(pairs)[q];
    const int sv = blk_src[b], nv = blk_ng[b];
    const int64_t nl_src = line_off[sv + 1] - line_off[sv];
    const int64_t nl_ng = line_off[nv + 1] - line_off[nv];
    int line = pr.x, ngl = pr.y;
    if (line < 0 || line >= nl_src) { *err = 1; line = 0; }
    if (ngl < 0 || ngl >= nl_ng) { *err = 2; ngl = 0; }
    key[r] = (uint32_t)(line_off[sv] + line);
    val[r] = ((uint32_t)nv << 16) | (uint32_t)ngl;
  }
}
void launch_expand_rows(const int32_t *d_pairs, const int64_t *d_blk_row_off, const int32_t *d_blk_src_view,
                        const int32_t *d_blk_ng_view, const int64_t *d_blk_pair_off, int n_blocks,
                        const int64_t *d_line_off, int64_t r_begin, int64_t r_end, uint32_t *d_key, uint32_t *d_val,
                        int *d_err, cudaStream_t s) {
  if (r_end <= r_begin) return;
  int grid = (int)((r_end - r_begin + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  expand_rows_kernel<<<grid, 256, 0, s>>>(d_pairs, d_blk_row_off, d_blk_src_view, d_blk_ng_view, d_blk_pair_off,
                                          n_blocks, d_line_off, r_begin, r_end, d_key, d_val, d_err);
}

// TriangulateImageExhaustiveMatch (base_line_triangulator.cc:111-136): every line of the neighbour.
__global__ void expand_exhaustive_kernel(const int64_t *__restrict__ blk_row_off, const int32_t *__restrict__ blk_src,
                                         const int32_t *__restrict__ blk_ng, int n_blocks,
                                         const int64_t *__restrict__ line_off, int64_t n_rows,
                                         uint32_t *__restrict__ key, uint32_t *__restrict__ val) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = n_blocks;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (blk_row_off[mid] <= r) lo = mid; else hi = mid;
    }
    const int b = lo;
    const int64_t q = r - blk_row_off[b];
    const int sv = blk_src[b], nv = blk_ng[b];
    const int64_t nl_ng = line_off[nv + 1] - line_off[nv];
    key[r] = (uint32_t)(line_off[sv] + q / nl_ng);
    val[r] = ((uint32_t)nv << 16) | (uint32_t)(q % nl_ng);
  }
}
void launch_expand_exhaustive(const int64_t *d_blk_row_off, const int32_t *d_blk_src_view,
                              const int32_t *d_blk_ng_view, int n_blocks, const int64_t *d_line_off, int64_t n_rows,
                              uint32_t *d_key, uint32_t *d_val, cudaStream_t s) {
  if (n_rows == 0) return;
  int grid = (int)((n_rows + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  expand_exhaustive_kernel<<<grid, 256, 0, s>>>(d_blk_row_off, d_blk_src_view, d_blk_ng_view, n_blocks, d_line_off,
                                                n_rows, d_key, d_val);
}

// Row range of every node in [node_lo, node_hi] from the node-sorted keys of one group (rows
// [row_base, row_base + n_rows) of the run); off[n] is a row index of the whole run.
__global__ void node_offsets_kernel(const uint32_t *__restrict__ key, int64_t n_rows, int64_t row_base,
                                    int64_t node_lo, int64_t node_hi, uint32_t *__restrict__ off,
                                    unsigned int *max_rows) {
  const int64_t n = node_lo + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (n > node_hi) return;
  int64_t lo = 0, hi = n_rows; // lower_bound(key, n)
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (key[mid] < (uint32_t)n) lo = mid + 1; else hi = mid;
  }
  off[n] = (uint32_t)(row_base + lo);
  if (n < node_hi) {
    int64_t lo2 = lo, hi2 = n_rows;
    while (lo2 < hi2) {
      const int64_t mid = (lo2 + hi2) >> 1;
      if (key[mid] < (uint32_t)(n + 1)) lo2 = mid + 1; else hi2 = mid;
    }
    const unsigned int cnt = (unsigned int)(lo2 - lo);
    if (cnt) atomicMax(max_rows, cnt);
  }
}
void launch_node_offsets(const uint32_t *d_sorted_key, int64_t n_rows, int64_t row_base, int64_t node_lo,
                         int64_t node_hi, uint32_t *d_node_row_off, unsigned int *d_max_rows, cudaStream_t s) {
  const int grid = (int)((node_hi - node_lo + 1 + 255) / 256);
  node_offsets_kernel<<<grid, 256, 0, s>>>(d_sorted_key, n_rows, row_base, node_lo, node_hi, d_node_row_off,
                                           d_max_rows);
}

// ------------------------------------------------------------------------------------------------
// Node-major rows by a per-view stable counting sort. The rows of a view are contiguous in flat order and its nodes are
// contiguous (line_off), so "stable sort by node id" is a stable partition of each view's rows by local line id. A view's
// rows are cut into tiles of kRowSortTile rows (never straddling a view); each tile histograms its lines (row_count),
// an exclusive prefix over the tiles of every (view, line) gives each tile's slot per line and the node row offsets
// (row_scan), and each tile writes its rows to their slots in row order (row_scatter). The result is the one a stable
// sort gives: d_key2/d_val2 and node_row_off byte for byte as the radix-sort path (expand_rows -> sort -> node_offsets).
static constexpr int kRowSortThreads = 256;
static constexpr int kRowSortWarps = kRowSortThreads / 32;
static constexpr int kRowSortSlice = kRowSortTile / kRowSortWarps; // contiguous rows per warp in row_scatter

// Per view i of the shard (view vb + i): first row vrow[i] (vrow[nvs] = rows of the shard), first tile vtile[i] and
// first tile-table word vtab[i] (a view's table is [tile][max(L, 1)]). Views above kRowSortMaxLines get no tiles.
// One CTA for the whole shard; the host derives the same numbers from its copy of the block table.
__global__ void row_views_kernel(const int64_t *__restrict__ blk_row_off, const int32_t *__restrict__ blk_src, int nb,
                                 const int64_t *__restrict__ line_off, int vb, int nvs, int64_t *__restrict__ vrow,
                                 int32_t *__restrict__ vtile, int64_t *__restrict__ vtab) {
  typedef cub::BlockScan<int64_t, kRowSortThreads> Scan;
  __shared__ typename Scan::TempStorage ts;
  __shared__ int64_t carry[2];
  if (threadIdx.x == 0) carry[0] = carry[1] = 0;
  __syncthreads();
  auto first_row = [&](int v) { // row offset of the first block with src_view >= v
    int lo = 0, hi = nb;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (blk_src[mid] < v) lo = mid + 1; else hi = mid;
    }
    return blk_row_off[lo];
  };
  for (int i0 = 0; i0 <= nvs; i0 += kRowSortThreads) {
    const int i = i0 + threadIdx.x;
    int64_t nt = 0, nw = 0;
    if (i <= nvs) {
      const int64_t r0 = first_row(vb + i);
      vrow[i] = r0;
      if (i < nvs) {
        const int64_t L = line_off[vb + i + 1] - line_off[vb + i];
        if (L <= kRowSortMaxLines) {
          nt = (first_row(vb + i + 1) - r0 + kRowSortTile - 1) / kRowSortTile;
          nw = nt * (L > 0 ? L : 1);
        }
      }
    }
    int64_t et, ew, at, aw;
    Scan(ts).ExclusiveSum(nt, et, at);
    __syncthreads();
    Scan(ts).ExclusiveSum(nw, ew, aw);
    if (i <= nvs) {
      vtile[i] = (int32_t)(carry[0] + et);
      vtab[i] = carry[1] + ew;
    }
    __syncthreads();
    if (threadIdx.x == 0) { carry[0] += at; carry[1] += aw; }
    __syncthreads();
  }
}

struct RowTile { // the tile a CTA of row_count / row_scatter works on
  int64_t node0, r0, r1, tab; // first node of the view, rows [r0, r1), its table row
  int L, Lb, b0, i;           // lines of the view, table stride max(L, 1), block of row r0, view index
};
__device__ __forceinline__ void row_tile_of(int tile, const int64_t *__restrict__ blk_row_off, int nb,
                                            const int64_t *__restrict__ line_off, int vb, const int64_t *__restrict__ vrow,
                                            const int32_t *__restrict__ vtile, const int64_t *__restrict__ vtab, int i_lo,
                                            int i_hi, RowTile &rt) {
  __shared__ RowTile s_rt;
  if (threadIdx.x == 0) {
    int lo = i_lo, hi = i_hi; // largest view i with vtile[i] <= tile (views without tiles are skipped)
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (vtile[mid] <= tile) lo = mid; else hi = mid;
    }
    RowTile t;
    t.i = lo;
    t.node0 = line_off[vb + lo];
    t.L = (int)(line_off[vb + lo + 1] - t.node0);
    t.Lb = t.L > 0 ? t.L : 1;
    const int64_t k = tile - vtile[lo];
    t.r0 = vrow[lo] + k * kRowSortTile;
    t.r1 = min(t.r0 + kRowSortTile, vrow[lo + 1]);
    t.tab = vtab[lo] + k * t.Lb;
    int b = 0, bh = nb; // largest block b with blk_row_off[b] <= r0
    while (bh - b > 1) {
      const int mid = (b + bh) >> 1;
      if (blk_row_off[mid] <= t.r0) b = mid; else bh = mid;
    }
    t.b0 = b;
    s_rt = t;
  }
  __syncthreads();
  rt = s_rt;
}

// Histogram of the tile's local line ids into its table row; index validation and clamping as expand_rows_kernel.
__global__ void __launch_bounds__(kRowSortThreads)
row_count_kernel(const int32_t *__restrict__ pairs, const int64_t *__restrict__ blk_row_off,
                 const int32_t *__restrict__ blk_ng, const int64_t *__restrict__ blk_pair_off, int nb,
                 const int64_t *__restrict__ line_off, int vb, const int64_t *__restrict__ vrow,
                 const int32_t *__restrict__ vtile, const int64_t *__restrict__ vtab, int i_lo, int i_hi, int tile0,
                 uint32_t *__restrict__ tab, int *err) {
  extern __shared__ uint32_t hist[];
  RowTile rt;
  row_tile_of(tile0 + blockIdx.x, blk_row_off, nb, line_off, vb, vrow, vtile, vtab, i_lo, i_hi, rt);
  for (int b = threadIdx.x; b < rt.Lb; b += kRowSortThreads) hist[b] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  int b = rt.b0;
  for (int64_t rr = rt.r0; rr < rt.r1; rr += kRowSortThreads) {
    const int64_t r = rr + threadIdx.x;
    int bin = -1;
    if (r < rt.r1) {
      while (blk_row_off[b + 1] <= r) ++b;
      const int2 pr = reinterpret_cast<const int2 *>(pairs)[blk_pair_off[b] + (r - blk_row_off[b])];
      const int nv = blk_ng[b];
      const int64_t nl_ng = line_off[nv + 1] - line_off[nv];
      bin = pr.x;
      if (bin < 0 || bin >= rt.L) { *err = 1; bin = 0; }
      if (pr.y < 0 || pr.y >= nl_ng) *err = 2;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (__ffs(peers) - 1) == lane) atomicAdd(&hist[bin], (uint32_t)__popc(peers));
  }
  __syncthreads();
  for (int k = threadIdx.x; k < rt.Lb; k += kRowSortThreads) tab[rt.tab + k] = hist[k];
}

// Per view (one CTA): exclusive prefix of every line's counts over the view's tiles, in place, and the node row
// offsets of the view's lines (a block scan of the line totals from the view's first row). Largest node -> max_rows.
__global__ void __launch_bounds__(kRowSortThreads)
row_scan_kernel(const int64_t *__restrict__ line_off, int vb, int i_lo, const int64_t *__restrict__ vrow,
                const int32_t *__restrict__ vtile, const int64_t *__restrict__ vtab, uint32_t *__restrict__ tab,
                uint32_t *__restrict__ node_row_off, unsigned int *max_rows) {
  typedef cub::BlockScan<uint32_t, kRowSortThreads> Scan;
  __shared__ typename Scan::TempStorage ts;
  const int i = i_lo + blockIdx.x;
  const int64_t node0 = line_off[vb + i], L = line_off[vb + i + 1] - node0;
  // the group's last node boundary (also the first row of the next view: the same value as any writer of it)
  if (threadIdx.x == 0 && blockIdx.x == gridDim.x - 1) node_row_off[node0 + L] = (uint32_t)vrow[i + 1];
  if (L > kRowSortMaxLines) return; // radix-sort fallback view
  const int nt = vtile[i + 1] - vtile[i];
  uint32_t *tb = tab + vtab[i];
  uint32_t run = (uint32_t)vrow[i], mx = 0;
  for (int64_t l0 = 0; l0 < L; l0 += kRowSortThreads) {
    const int64_t l = l0 + threadIdx.x;
    uint32_t tot = 0;
    if (l < L) {
#pragma unroll 4
      for (int t = 0; t < nt; ++t) {
        const uint32_t c = tb[(int64_t)t * L + l];
        tb[(int64_t)t * L + l] = tot;
        tot += c;
      }
    }
    mx = max(mx, tot);
    uint32_t ex, agg;
    Scan(ts).ExclusiveSum(tot, ex, agg);
    if (l < L) node_row_off[node0 + l] = run + ex;
    run += agg;
    __syncthreads();
  }
  mx = __reduce_max_sync(0xffffffffu, mx);
  if ((threadIdx.x & 31) == 0 && mx) atomicMax(max_rows, mx);
}

// Rows of the tile to their slots. Warp w owns rows [r0 + w * kRowSortSlice, ...) of the tile: it counts its slice per
// line, the counts of the warps are combined in warp order on top of the tile's slot per line, and the warp then walks
// its slice again in row order, ranking equal lines inside each 32-row step with __match_any_sync.
__global__ void __launch_bounds__(kRowSortThreads)
row_scatter_kernel(const int32_t *__restrict__ pairs, const int64_t *__restrict__ blk_row_off,
                   const int32_t *__restrict__ blk_ng, const int64_t *__restrict__ blk_pair_off, int nb,
                   const int64_t *__restrict__ line_off, int vb, const int64_t *__restrict__ vrow,
                   const int32_t *__restrict__ vtile, const int64_t *__restrict__ vtab, int i_lo, int i_hi, int tile0,
                   const uint32_t *__restrict__ tab, const uint32_t *__restrict__ node_row_off,
                   uint32_t *__restrict__ key, uint32_t *__restrict__ val) {
  extern __shared__ uint32_t ctr[]; // [warp][Lb]: the warp's count per line, then its next slot per line
  RowTile rt;
  row_tile_of(tile0 + blockIdx.x, blk_row_off, nb, line_off, vb, vrow, vtile, vtab, i_lo, i_hi, rt);
  for (int k = threadIdx.x; k < kRowSortWarps * rt.Lb; k += kRowSortThreads) ctr[k] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t *wc = ctr + w * rt.Lb;
  const int64_t ws = rt.r0 + (int64_t)w * kRowSortSlice, we = min(ws + kRowSortSlice, rt.r1);
  int b = rt.b0;
  for (int64_t rr = ws; rr < we; rr += 32) {
    const int64_t r = rr + lane;
    int bin = -1;
    if (r < we) {
      while (blk_row_off[b + 1] <= r) ++b;
      bin = reinterpret_cast<const int2 *>(pairs)[blk_pair_off[b] + (r - blk_row_off[b])].x;
      if (bin < 0 || bin >= rt.L) bin = 0;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (__ffs(peers) - 1) == lane) wc[bin] += (uint32_t)__popc(peers);
    __syncwarp();
  }
  __syncthreads();
  for (int k = threadIdx.x; k < rt.Lb; k += kRowSortThreads) {
    // (a view without lines only has out-of-range rows, clamped to line 0: keep them inside the view's rows)
    uint32_t base = (k < rt.L ? node_row_off[rt.node0 + k] : (uint32_t)vrow[rt.i]) + (rt.L > 0 ? tab[rt.tab + k] : 0u);
    for (int ww = 0; ww < kRowSortWarps; ++ww) {
      const uint32_t c = ctr[ww * rt.Lb + k];
      ctr[ww * rt.Lb + k] = base;
      base += c;
    }
  }
  __syncthreads();
  b = rt.b0;
  const unsigned lt = (1u << lane) - 1u;
  for (int64_t rr = ws; rr < we; rr += 32) {
    const int64_t r = rr + lane;
    int bin = -1, nv = 0, ngl = 0;
    if (r < we) {
      while (blk_row_off[b + 1] <= r) ++b;
      const int2 pr = reinterpret_cast<const int2 *>(pairs)[blk_pair_off[b] + (r - blk_row_off[b])];
      nv = blk_ng[b];
      const int64_t nl_ng = line_off[nv + 1] - line_off[nv];
      bin = pr.x;
      ngl = pr.y;
      if (bin < 0 || bin >= rt.L) bin = 0;
      if (ngl < 0 || ngl >= nl_ng) ngl = 0;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    const uint32_t pos = bin >= 0 ? wc[bin] + (uint32_t)__popc(peers & lt) : 0u;
    __syncwarp();
    if (bin >= 0 && (__ffs(peers) - 1) == lane) wc[bin] += (uint32_t)__popc(peers);
    __syncwarp();
    if (bin >= 0) {
      key[pos] = (uint32_t)(rt.node0 + bin);
      val[pos] = ((uint32_t)nv << 16) | (uint32_t)ngl;
    }
  }
}

size_t row_scatter_smem_bytes(int max_lines) { return (size_t)kRowSortWarps * 4 * (size_t)std::max(max_lines, 1); }

void launch_row_views(const int64_t *d_blk_row_off, const int32_t *d_blk_src_view, int n_blocks,
                      const int64_t *d_line_off, int vb, int n_views, int64_t *d_vrow, int32_t *d_vtile, int64_t *d_vtab,
                      cudaStream_t s) {
  row_views_kernel<<<1, kRowSortThreads, 0, s>>>(d_blk_row_off, d_blk_src_view, n_blocks, d_line_off, vb, n_views,
                                                  d_vrow, d_vtile, d_vtab);
}

cudaError_t launch_row_sort(const int32_t *d_pairs, const int64_t *d_blk_row_off, const int32_t *d_blk_ng_view,
                            const int64_t *d_blk_pair_off, int n_blocks, const int64_t *d_line_off, int vb,
                            const int64_t *d_vrow, const int32_t *d_vtile, const int64_t *d_vtab, int i_lo, int i_hi,
                            int tile0, int n_tiles, int max_lines, uint32_t *d_tab, uint32_t *d_node_row_off,
                            unsigned int *d_max_rows, uint32_t *d_key, uint32_t *d_val, int *d_err, cudaStream_t s) {
  if (i_hi <= i_lo) return cudaSuccess;
  if (n_tiles > 0)
    row_count_kernel<<<n_tiles, kRowSortThreads, 4 * std::max(max_lines, 1), s>>>(
        d_pairs, d_blk_row_off, d_blk_ng_view, d_blk_pair_off, n_blocks, d_line_off, vb, d_vrow, d_vtile, d_vtab, i_lo,
        i_hi, tile0, d_tab, d_err);
  row_scan_kernel<<<i_hi - i_lo, kRowSortThreads, 0, s>>>(d_line_off, vb, i_lo, d_vrow, d_vtile, d_vtab, d_tab,
                                                          d_node_row_off, d_max_rows);
  if (n_tiles > 0) {
    const size_t smem = row_scatter_smem_bytes(max_lines);
    if (smem > 48 * 1024) {
      const cudaError_t e = cudaFuncSetAttribute(row_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
    }
    row_scatter_kernel<<<n_tiles, kRowSortThreads, smem, s>>>(d_pairs, d_blk_row_off, d_blk_ng_view, d_blk_pair_off,
                                                              n_blocks, d_line_off, vb, d_vrow, d_vtile, d_vtab, i_lo,
                                                              i_hi, tile0, d_tab, d_node_row_off, d_key, d_val);
  }
  return cudaGetLastError();
}

// valid_edges_ (global_line_triangulator.cc:130-142) in compact, node-major, candidate-ordered form.
__global__ void extract_nvalid_kernel(const NodeRecord *__restrict__ nodes, int64_t node_begin, int64_t n,
                                      uint32_t *__restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = (uint32_t)nodes[node_begin + i].n_valid;
  if (i == n) out[i] = 0;
}
__global__ void compact_edges_kernel(const uint8_t *__restrict__ row_state, const uint32_t *__restrict__ row_ng,
                                     const uint32_t *__restrict__ node_row_off, const uint32_t *__restrict__ edge_off,
                                     int64_t node_begin, int64_t n, int ns, uint32_t *__restrict__ edge_ng) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / 32;
  if (i >= n) return;
  const int64_t q0 = (int64_t)node_row_off[node_begin + i] * ns, q1 = (int64_t)node_row_off[node_begin + i + 1] * ns;
  uint32_t base = edge_off[i];
  if (edge_off[i + 1] == base) return;
  for (int64_t qb = q0; qb < q1; qb += 32) { // q = row * ns + slot: candidate order
    const int64_t q = qb + lane;
    const bool v = (q < q1) && row_state[q] == 2;
    const unsigned m = __ballot_sync(0xffffffffu, v);
    if (v) edge_ng[base + __popc(m & ((1u << lane) - 1u))] = row_ng[q / ns];
    base += __popc(m);
  }
}
// Valid connections of one pipeline group, right after the group's node kernel: global offsets (the groups before it are
// done: their totals are on the device) and compact (neighbour view << 16 | line) entries in candidate order. One warp
// per node. (Writing the caller's page-locked result buffers from here over PCIe was measured: 0.25 ms SLOWER per step
// than one device-to-host copy after the run.)
__global__ void group_edges_kernel(const uint8_t *__restrict__ row_state, const uint32_t *__restrict__ row_ng,
                                   const uint32_t *__restrict__ node_row_off, const uint32_t *__restrict__ local_off,
                                   unsigned int *__restrict__ totals, int g, int64_t shard_node_begin, int64_t node_lo, int64_t n,
                                   int ns, uint32_t *__restrict__ edge_off, uint32_t *__restrict__ edge_ng) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / 32;
  if (i >= n) return;
  uint32_t before = 0;
  for (int k = 0; k < g; ++k) before += totals[k];
  const uint32_t lo = local_off[i], hi = local_off[i + 1];
  uint32_t base = before + lo;
  if (lane == 0) {
    edge_off[node_lo - shard_node_begin + i] = base;
    if (i == n - 1) {
      edge_off[node_lo - shard_node_begin + n] = before + local_off[n];
      totals[g] = local_off[n];
    }
  }
  if (hi == lo) return;
  const int64_t q0 = (int64_t)node_row_off[node_lo + i] * ns, q1 = (int64_t)node_row_off[node_lo + i + 1] * ns;
  for (int64_t qb = q0; qb < q1; qb += 32) { // q = row * ns + slot: candidate order
    const int64_t q = qb + lane;
    const bool v = (q < q1) && row_state[q] == 2;
    const unsigned m = __ballot_sync(0xffffffffu, v);
    if (v) edge_ng[base + __popc(m & ((1u << lane) - 1u))] = row_ng[q / ns];
    base += __popc(m);
  }
}
void launch_group_edges(const uint8_t *row_state, const uint32_t *row_ng, const uint32_t *node_row_off,
                        const uint32_t *local_off, unsigned int *totals, int g, int64_t shard_node_begin, int64_t node_lo,
                        int64_t n, int ns, uint32_t *edge_off, uint32_t *edge_ng, cudaStream_t s) {
  if (n <= 0) return;
  group_edges_kernel<<<(int)((n * 32 + 255) / 256), 256, 0, s>>>(row_state, row_ng, node_row_off, local_off, totals, g,
                                                                 shard_node_begin, node_lo, n, ns, edge_off, edge_ng);
}
// directed (src node, dst node) pairs of the compact edge list
__global__ void edge_pairs_kernel(const uint32_t *__restrict__ edge_off, const uint32_t *__restrict__ edge_ng,
                                  const int64_t *__restrict__ line_off, int64_t node_begin, int64_t n_nodes,
                                  int64_t n_edges, int64_t *__restrict__ out) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n_edges) return;
  int64_t lo = 0, hi = n_nodes; // largest i with edge_off[i] <= e
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (edge_off[mid] <= (uint32_t)e) lo = mid; else hi = mid;
  }
  const uint32_t ng = edge_ng[e];
  out[2 * e] = node_begin + lo;
  out[2 * e + 1] = line_off[ng >> 16] + (ng & 0xffffu);
}
void launch_edge_pairs(const uint32_t *edge_off, const uint32_t *edge_ng, const int64_t *line_off,
                       int64_t node_begin, int64_t n_nodes, int64_t n_edges, int64_t *out, cudaStream_t s) {
  if (n_edges <= 0) return;
  edge_pairs_kernel<<<(int)((n_edges + 255) / 256), 256, 0, s>>>(edge_off, edge_ng, line_off, node_begin, n_nodes,
                                                                 n_edges, out);
}
void launch_extract_nvalid(const NodeRecord *nodes, int64_t node_begin, int64_t n, uint32_t *out, cudaStream_t s) {
  extract_nvalid_kernel<<<(int)((n + 1 + 255) / 256), 256, 0, s>>>(nodes, node_begin, n, out);
}
void launch_compact_edges_only(const uint8_t *row_state, const uint32_t *row_ng, const uint32_t *node_row_off,
                               const uint32_t *edge_off, int64_t node_begin, int64_t n, int ns, uint32_t *edge_ng,
                               cudaStream_t s) {
  if (n <= 0) return;
  compact_edges_kernel<<<(int)((n * 32 + 255) / 256), 256, 0, s>>>(row_state, row_ng, node_row_off, edge_off,
                                                                   node_begin, n, ns, edge_ng);
}

// valid connections as (ng_img_id, ng_line_id) int32 pairs + int64 node offsets, ready for the caller's buffer
__global__ void edges_for_host_kernel(const uint32_t *__restrict__ edge_off, const uint32_t *__restrict__ edge_ng,
                                      const int32_t *__restrict__ img_ids, int64_t n_nodes_shard, int64_t n_edges,
                                      int64_t node_begin, int64_t n_nodes_total, int64_t *__restrict__ node_off,
                                      int32_t *__restrict__ pairs) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < n_edges) {
    const uint32_t ng = edge_ng[t];
    pairs[2 * t] = img_ids[ng >> 16];
    pairs[2 * t + 1] = (int32_t)(ng & 0xffffu);
  }
  if (t <= n_nodes_total) {
    int64_t v = 0;
    if (t >= node_begin && t <= node_begin + n_nodes_shard) v = edge_off[t - node_begin];
    else if (t > node_begin + n_nodes_shard) v = n_edges;
    node_off[t] = v;
  }
}
void launch_edges_for_host(const uint32_t *edge_off, const uint32_t *edge_ng, const int32_t *img_ids,
                           int64_t n_nodes_shard, int64_t n_edges, int64_t node_begin, int64_t n_nodes_total,
                           int64_t *node_off, int32_t *pairs, cudaStream_t s) {
  const int64_t n = (n_edges > n_nodes_total + 1) ? n_edges : n_nodes_total + 1;
  edges_for_host_kernel<<<(int)((n + 255) / 256), 256, 0, s>>>(edge_off, edge_ng, img_ids, n_nodes_shard, n_edges,
                                                               node_begin, n_nodes_total, node_off, pairs);
}

// ---- scene preparation: the 2D segments as the kernels read them (add_halfpix, base_line_triangulator.cc:32-43) and the
// view of every node, derived on the device from what lm_scene_upload copied ------------------------------------------
__global__ void scene_prepare_kernel(const double *__restrict__ segs_raw, int64_t n_nodes, double add,
                                     const int64_t *__restrict__ line_off, int n_views, double *__restrict__ segs,
                                     uint16_t *__restrict__ node_view) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < 4 * n_nodes) segs[i] = segs_raw[i] + add;
  if (i < n_nodes && node_view) {
    int lo = 0, hi = n_views; // largest v with line_off[v] <= i
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (line_off[mid] <= i) lo = mid; else hi = mid;
    }
    node_view[i] = (uint16_t)lo;
  }
}
void launch_scene_prepare(const double *segs_raw, int64_t n_nodes, double add, const int64_t *line_off, int n_views,
                          double *segs, uint16_t *node_view, cudaStream_t s) {
  if (n_nodes <= 0) return;
  scene_prepare_kernel<<<(int)((4 * n_nodes + 255) / 256), 256, 0, s>>>(segs_raw, n_nodes, add, line_off, n_views, segs, node_view);
}

// ---- multi-GPU exchange: one fixed-size message per rank (SURVEY.md 8e: "one all-gather of per-node results") ----
// message = [int64 n_edges, int64 n_nodes] | NodeRecord[max_nodes] | (uint32 src_node, uint32 dst_node)[cap_edges]
__global__ void gather_pack_kernel(const NodeRecord *__restrict__ nodes, int64_t node_begin, int64_t n_nodes,
                                   int64_t max_nodes, const uint32_t *__restrict__ edge_off,
                                   const uint32_t *__restrict__ edge_ng, const int64_t *__restrict__ line_off,
                                   int64_t cap_edges, char *__restrict__ msg) {
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  const int64_t ne = n_nodes > 0 ? (int64_t)edge_off[n_nodes] : 0;
  if (tid == 0) { reinterpret_cast<int64_t *>(msg)[0] = ne; reinterpret_cast<int64_t *>(msg)[1] = n_nodes; }
  const uint4 *src = reinterpret_cast<const uint4 *>(nodes + node_begin);
  uint4 *dst = reinterpret_cast<uint4 *>(msg + 16);
  const int64_t nv = n_nodes * (int64_t)(sizeof(NodeRecord) / 16);
  for (int64_t i = tid; i < nv; i += nth) dst[i] = src[i];
  uint2 *ed = reinterpret_cast<uint2 *>(msg + 16 + max_nodes * (int64_t)sizeof(NodeRecord));
  const int64_t nc = ne < cap_edges ? ne : cap_edges;
  for (int64_t e = tid; e < nc; e += nth) {
    int64_t lo = 0, hi = n_nodes; // largest i with edge_off[i] <= e
    while (hi - lo > 1) {
      const int64_t mid = (lo + hi) >> 1;
      if (edge_off[mid] <= (uint32_t)e) lo = mid; else hi = mid;
    }
    const uint32_t ng = edge_ng[e];
    ed[e] = make_uint2((uint32_t)(node_begin + lo), (uint32_t)(line_off[ng >> 16] + (ng & 0xffffu)));
  }
}
// all ranks' messages -> node records in place, directed edges appended in rank order as int64 pairs;
// scal[0] = total edges, scal[1] = 1 when some rank had more edges than the message holds
__global__ void gather_unpack_kernel(const char *__restrict__ msgs, int world, const int64_t *__restrict__ rank_node_begin,
                                     int64_t max_nodes, int64_t cap_edges, int64_t msg_bytes,
                                     NodeRecord *__restrict__ nodes, int64_t *__restrict__ edges,
                                     int64_t *__restrict__ scal) {
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  int64_t ebase = 0;
  bool over = false;
  for (int r = 0; r < world; ++r) {
    const char *m = msgs + r * msg_bytes;
    int64_t ne = reinterpret_cast<const int64_t *>(m)[0];
    const int64_t nn = reinterpret_cast<const int64_t *>(m)[1];
    if (ne > cap_edges) { over = true; ne = cap_edges; }
    const uint4 *src = reinterpret_cast<const uint4 *>(m + 16);
    uint4 *dst = reinterpret_cast<uint4 *>(nodes + rank_node_begin[r]);
    const int64_t nv = nn * (int64_t)(sizeof(NodeRecord) / 16);
    for (int64_t i = tid; i < nv; i += nth) dst[i] = src[i];
    const uint2 *ed = reinterpret_cast<const uint2 *>(m + 16 + max_nodes * (int64_t)sizeof(NodeRecord));
    for (int64_t e = tid; e < ne; e += nth) {
      const uint2 v = ed[e];
      edges[2 * (ebase + e)] = (int64_t)v.x;
      edges[2 * (ebase + e) + 1] = (int64_t)v.y;
    }
    ebase += ne;
  }
  if (tid == 0) { scal[0] = ebase; scal[1] = over ? 1 : 0; }
}
void launch_gather_pack(const NodeRecord *nodes, int64_t node_begin, int64_t n_nodes, int64_t max_nodes,
                        const uint32_t *edge_off, const uint32_t *edge_ng, const int64_t *line_off, int64_t cap_edges,
                        char *msg, cudaStream_t s) {
  gather_pack_kernel<<<148 * 4, 256, 0, s>>>(nodes, node_begin, n_nodes, max_nodes, edge_off, edge_ng, line_off, cap_edges, msg);
}
void launch_gather_unpack(const char *msgs, int world, const int64_t *rank_node_begin, int64_t max_nodes, int64_t cap_edges,
                          int64_t msg_bytes, NodeRecord *nodes, int64_t *edges, int64_t *scal, cudaStream_t s) {
  gather_unpack_kernel<<<148 * 4, 256, 0, s>>>(msgs, world, rank_node_begin, max_nodes, cap_edges, msg_bytes, nodes, edges, scal);
}

// run_clustering edge weight (global_line_triangulator.cc:263-288): LineLinker3d::compute_score of the
// two best lines under set_to_spatial_merging().
__global__ void edge_weights_kernel(const __grid_constant__ EdgeParams p) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= p.n) return;
  const NodeRecord &a = p.nodes[p.edges[2 * e]];
  const NodeRecord &b = p.nodes[p.edges[2 * e + 1]];
  seg<vec3<double>> l1, l2;
  l1.s = mk3(a.line[0], a.line[1], a.line[2]); l1.e = mk3(a.line[3], a.line[4], a.line[5]);
  l2.s = mk3(b.line[0], b.line[1], b.line[2]); l2.e = mk3(b.line[3], b.line[4], b.line[5]);
  const double unc = smin(a.line[8], b.line[8]);
  p.weight[e] = linker_score<double, vec3<double>>(p.l3d, l1, l2, unc, true, a.line[6], a.line[7]);
}
void launch_edge_weights(const EdgeParams &p, cudaStream_t s) {
  if (p.n <= 0) return;
  const int grid = (int)((p.n + 127) / 128);
  edge_weights_kernel<<<grid, 128, 0, s>>>(p);
}

} // namespace lm
