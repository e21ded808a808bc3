/*
 * fuel_oracle.h -- CPU restatement of FUEL's per-replan hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in fuel_b200/ may include, link or call this.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs use it, and only as the checker / the timed CPU baseline.
 *
 * PARITY STATUS: pinned against the reference's own code for everything except two third-party algorithms.
 * The reference (HKUST-Aerial-Robotics/FUEL @ 662dd23) ships no golden vectors or unit tests for this path (SURVEY.md
 * section 4) and its build needs ROS1, Eigen3, PCL, NLopt (absent, no network) -- but its hot-path sources compile
 * UNMODIFIED from /root/reference against the interface stand-ins of oracle/ref_standin/ (oracle/Makefile ->
 * oracle/_ref/libfuel_ref.so): plan_env/src/{sdf_map,raycast}.cpp, bspline_opt/src/bspline_optimizer.cpp,
 * active_perception/src/{frontier_finder,perception_utils}.cpp.  tests/test_oracle_refpin.py compares this oracle
 * with that code bit for bit (ESDF all modes, inflation, fusion, getDistWithGrad, RayCaster, combineCost for every
 * term combination, frontier search / split / flags, viewpoint sampling, isFrontierCovered).
 * "parity unpinned" remains for the third-party arithmetic reconstructed from published algorithms (the stand-ins
 * call these very functions, so the comparison does not cover them):
 *   - PCL >= 1.7 VoxelGrid<PointXYZ>::applyFilter   (frontier_finder.cpp:757-774)  -> orc_voxelgrid_f32
 *   - Eigen 3.3 EigenSolver<Matrix2d>               (frontier_finder.cpp:202-213)  -> orc_eigen_sym2x2
 * and for NLopt's iterate sequence (not restated; orc_optimize_batch is the twin of OUR solver).
 *
 * All file:line citations are relative to /root/reference/fuel_planner/.
 */
#ifndef FUEL_ORACLE_H
#define FUEL_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Grid geometry: plan_env/include/plan_env/sdf_map.h:86-105 (struct MapParam). */
typedef struct {
  int32_t n[3];       /* map_voxel_num_ (x,y,z); address = x*ny*nz + y*nz + z, sdf_map.h:145-147 */
  double res;         /* resolution_ */
  double origin[3];   /* map_origin_ = map_min_boundary_ */
  double box_mind[3]; /* box_mind_ (exploration box, metres) */
  double box_maxd[3]; /* box_maxd_ */
  double map_size[3]; /* map_size_: map_max_boundary_ = origin + map_size_ (sdf_map.cpp:34-39); all zero = n*res */
} OrcGrid;

/* Occupancy tri-state, sdf_map.h:32 and :194-200 (getOccupancy). */
enum { ORC_UNKNOWN = 0, ORC_FREE = 1, ORC_OCCUPIED = 2 };

/* ---- index helpers (sdf_map.h:127-237) -------------------------------------------- */
void orc_pos_to_index(const OrcGrid* g, const double pos[3], int32_t id[3]);
void orc_index_to_pos(const OrcGrid* g, const int32_t id[3], double pos[3]);
int orc_is_in_map_pos(const OrcGrid* g, const double pos[3]);
/* tri-state from log-odds, sdf_map.h:194-200 */
void orc_tristate_from_logodds(const double* logodds, int64_t n, double clamp_min_log,
                               double min_occupancy_log, uint8_t* tri);

/* ---- ESDF: sdf_map.cpp:116-150 (fillESDF), :152-241 (updateESDF3d) ------------------
 * inflate : occupancy_buffer_inflate_ (char {0,1})
 * tri     : tri-state derived from occupancy_buffer_ (only "== UNKNOWN" is consulted, which
 *           is exactly the reference's `occupancy_buffer_[adr] < clamp_min_log_ - 1e-3`);
 *           may be NULL when optimistic != 0
 * bmin/bmax : local_bound_min_/max_ (inclusive)
 * dist    : distance_buffer_ (written inside the box only)
 * dist_neg: distance_buffer_neg_ (only touched when signed_dist != 0; may be NULL otherwise)
 * tmp1/tmp2 : tmp_buffer1_/2_ scratch of full volume size
 * threads : 1 = the reference's single thread; >1 = OpenMP over independent lines (the
 *           "all host cores" baseline; identical results, lines are independent)
 */
void orc_update_esdf3d(const OrcGrid* g, const int8_t* inflate, const uint8_t* tri,
                       const int32_t bmin[3], const int32_t bmax[3], int optimistic,
                       int signed_dist, double* dist, double* dist_neg, double* tmp1,
                       double* tmp2, int threads);

/* clearAndInflateLocalMap, sdf_map.cpp:364-472 (the step right before updateESDF3d; SURVEY 8f rank 2).
 * tri     : getOccupancy() of occupancy_buffer_ (in/out: the virtual ceiling writes clamp_max_log_,
 *           i.e. OCCUPIED, at z = ceil_id, :463-470)
 * inflate : occupancy_buffer_inflate_ (in/out)
 * inf_step: ceil(obstacles_inflation_ / resolution_) (:436); the stamp is (2*inf_step+1)^3 ("all inflate",
 *           sdf_map.h:257-264).  The linear-address-only bounds check of :452-458 (stamps wrap across
 *           rows at the map faces, SURVEY H9) is reproduced as written.
 * ceil_id : floor((virtual_ceil_height_ - origin_z) * resolution_inv_), or < 0 to disable (:462) */
void orc_clear_and_inflate(const OrcGrid* g, uint8_t* tri, int8_t* inflate, const int32_t bmin[3],
                           const int32_t bmax[3], int inf_step, int ceil_id);

/* ---- occupancy fusion: sdf_map.cpp:243-345 inputPointCloud (SURVEY 8f rank 3); fuel_oracle_fusion.c ---- */
typedef struct {
  double p_hit, p_miss, p_min, p_max, p_occ; /* probabilities; logit()ed like sdf_map.cpp:36-47 */
  double max_ray_length, local_bound_inflate;
} OrcFusionParams;
typedef struct {
  int16_t *count_hit, *count_miss; /* md_->count_hit_/count_miss_ (short) */
  int8_t* flag_rayend;             /* md_->flag_rayend_ (char, initialised -1, sdf_map.cpp:71) */
  int8_t raycast_num;              /* md_->raycast_num_ (char counter) */
  int32_t reset_updated_box;       /* md_->reset_updated_box_ */
  double update_min[3], update_max[3];
} OrcFusionState;
void orc_fusion_state_init(OrcFusionState* st, int64_t nvox);
void orc_fusion_state_free(OrcFusionState* st);
/* logodds = occupancy_buffer_ (in/out); points = float32 xyz; local_bound_min/max = md_->local_bound_min_/max_ out */
void orc_input_point_cloud(const OrcGrid* g, const OrcFusionParams* fp, OrcFusionState* st, double* logodds,
                           const float* points, int32_t point_num, const double camera_pos[3],
                           int32_t local_bound_min[3], int32_t local_bound_max[3]);

/* MapROS::proessDepthImage, plan_env/src/map_ros.cpp:176-215: depth image (uint16, rows x cols, row-major) ->
 * world points (float32 xyz, as stored in pcl::PointXYZ), in the order the reference emits them.  R = row-major
 * camera_q_.toRotationMatrix().  Returns proj_points_cnt.  The zero test reads the pixel skip_pixel to the right of
 * the one whose depth is used (row_ptr is advanced first, :190-198) -- reproduced. */
typedef struct {
  double fx, fy, cx, cy;
  double k_depth_scaling_factor, depth_filter_maxdist, depth_filter_mindist;
  int32_t depth_filter_margin, skip_pixel;
} OrcCameraParams;
int32_t orc_process_depth_image(const OrcCameraParams* cp, const uint16_t* depth, int32_t rows, int32_t cols,
                                const double R[9], const double camera_pos[3], float* points_out);

int32_t orc_raycast_ids(const OrcGrid* g, const double start[3], const double end[3], int32_t* ids, int32_t max);
double orc_intbound(double s, double ds);

/* sdf_map.cpp:497-536 getDistWithGrad (via EDTEnvironment::evaluateEDTWithGrad,
 * edt_environment.cpp:78-87).  dist_buf = distance_buffer_. */
double orc_dist_with_grad(const OrcGrid* g, const double* dist_buf, const double pos[3],
                          double grad[3]);
void orc_dist_with_grad_batch(const OrcGrid* g, const double* dist_buf, int64_t n,
                              const double* pos, double* dist, double* grad);

/* ---- Frontier: active_perception/src/frontier_finder.cpp ---------------------------- */
typedef struct {
  int32_t cluster_min;     /* frontier/cluster_min     (:29)  */
  double cluster_size_xy;  /* frontier/cluster_size_xy (:30)  */
  int32_t down_sample;     /* frontier/down_sample     (:38)  */
  double min_z;            /* the literal 0.4 at :152         */
  int32_t cell_order;      /* 0 = BFS order (the reference, :139-156);
                              1 = canonical: each cluster's cells_ re-sorted by ascending
                                  address before computeFrontierInfo (what the GPU emits) */
} OrcFrontierParams;

typedef struct OrcFrontierResult OrcFrontierResult;

/* searchFrontiers (:54-121) restricted to its stateless core: the sweep over the search
 * box, expandFrontier (:123-164), computeFrontierInfo (:374-390), downsample (:757-774),
 * splitLargeFrontiers / splitHorizontally (:166-242).
 * flag      : frontier_flag_ (in/out, char per voxel)
 * upd_min/upd_max : the updated box (metres) as returned by getUpdatedBox
 * Removal of changed stored frontiers (:65-92) is list bookkeeping that lives in the
 * host-side FrontierFinder mirror; see orc_frontier_is_changed. */
OrcFrontierResult* orc_frontier_search(const OrcGrid* g, const uint8_t* tri, int8_t* flag,
                                       const double upd_min[3], const double upd_max[3],
                                       const OrcFrontierParams* p);
int32_t orc_frontier_count(const OrcFrontierResult* r);
int32_t orc_frontier_num_cells(const OrcFrontierResult* r, int32_t i);
int32_t orc_frontier_num_filtered(const OrcFrontierResult* r, int32_t i);
/* addr: n cells (toAddress); filtered: m*3 doubles; avg[3]; bmin[3]; bmax[3] */
void orc_frontier_get(const OrcFrontierResult* r, int32_t i, int32_t* addr, double* filtered,
                      double avg[3], double bmin[3], double bmax[3]);
void orc_frontier_free(OrcFrontierResult* r);
/* isFrontierChanged (:365-372) on a list of cell addresses. */
int orc_frontier_is_changed(const OrcGrid* g, const uint8_t* tri, const int32_t* addr, int32_t n);
/* the per-voxel predicate knownfree && isNeighborUnknown (:862-881) */
int orc_is_frontier_cell(const OrcGrid* g, const uint8_t* tri, const int32_t id[3]);
/* principal axis of a symmetric 2x2 matrix under the reconstructed Eigen 3.3
 * EigenSolver convention (:202-213); exposed for its own tests */
void orc_principal_axis_2x2(double a, double b, double d, double pc[2]);
/* the two third-party reconstructions on their own (also used by oracle/ref_standin, see fuel_oracle.c) */
void orc_eigen_sym2x2(double a, double b, double d, double vals[2], double vecs[2][2]);
int32_t orc_voxelgrid_f32(const float* pts, int32_t n, float leaf, float* out);

/* ---- viewpoint sampling (SURVEY 8f rank 4); fuel_oracle_viewpoints.c ------------------------------- */
typedef struct {
  double candidate_rmin, candidate_rmax; /* frontier/candidate_rmin, rmax (frontier_finder.cpp:35-36) */
  int32_t candidate_rnum;                /* frontier/candidate_rnum (:37) */
  double candidate_dphi;                 /* frontier/candidate_dphi (:34) */
  double min_candidate_clearance;        /* frontier/min_candidate_clearance (:33) */
  double top_angle, left_angle, right_angle, max_dist; /* perception_utils params (perception_utils.cpp:7-10) */
} OrcViewParams;
int32_t orc_viewpoint_candidates(const OrcViewParams* vp, double* off_xy, int32_t max);
int32_t orc_sample_viewpoints(const OrcGrid* g, const uint8_t* tri, const int8_t* inflate, const OrcViewParams* vp,
                              const double average[3], const double* cells, int32_t n_cells, double* cand_pos,
                              double* cand_yaw, int32_t* cand_visib, uint8_t* cand_border);
int32_t orc_frontier_changed_count(const OrcGrid* g, const uint8_t* tri, const int32_t* addr, int32_t n);

/* ---- B-spline cost: bspline_opt/src/bspline_optimizer.cpp ---------------------------- */
enum {
  ORC_SMOOTHNESS = 1 << 0, ORC_DISTANCE = 1 << 1, ORC_FEASIBILITY = 1 << 2,
  ORC_START = 1 << 3, ORC_END = 1 << 4, ORC_GUIDE = 1 << 5, ORC_WAYPOINTS = 1 << 6,
  ORC_VIEWCONS = 1 << 7, ORC_MINTIME = 1 << 8
}; /* :10-23 */

typedef struct {
  double ld_smooth, ld_dist, ld_feasi, ld_start, ld_end, ld_guide, ld_waypt, ld_view, ld_time;
  double dist0, max_vel, max_acc;
  int32_t order; /* order_ = bspline_degree_ (3) */
  double wnl;    /* wnl_ (optimization/wnl, :44): weight of the parallel part of calcViewCost */
} OrcOptParams;   /* setParam :25-57 */

#define ORC_MAX_PTS 64
typedef struct {
  double pt_dist;          /* :136-140 */
  double knot_span;        /* knot_span_ (used when MINTIME is off) */
  double start[3][3];      /* start_state_ pos, vel, acc */
  double end[3][3];        /* end_state_ */
  int32_t n_end;           /* end_state_.size() in 1..3 */
  double time_lb;          /* time_lb_ */
  int32_t n_guide;         /* guide_pts_.size() (N - 2*order) */
  double guide[ORC_MAX_PTS][3];
  int32_t n_waypt;
  double waypt[ORC_MAX_PTS][3];
  int32_t waypt_idx[ORC_MAX_PTS];
  double view_pt[3];       /* view_cons_.pt_  (setViewConstraint :91-93; active_perception/traj_visibility.h:18-24) */
  double view_dir[3];      /* view_cons_.dir_ (length = safe distance) */
  int32_t view_idx;        /* view_cons_.idx_; < 0: no constraint set */
} OrcTrajConst;

/* combineCost (:518-647) for dim_ == 3.  x has 3N (+1 if MINTIME) entries. */
void orc_combine_cost(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                      const OrcTrajConst* tc, int32_t n_pts, int32_t cost_mask,
                      const double* x, double* f, double* grad);
/* B independent evaluations; threads>1 -> OpenMP over trajectories */
void orc_combine_cost_batch(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                            const OrcTrajConst* tc /*[B]*/, int32_t n_pts, int32_t cost_mask,
                            int32_t B, const double* x /*[B][nvar]*/, double* f /*[B]*/,
                            double* grad /*[B][nvar]*/, int threads);
/* pt_dist_ as computed in optimize(), :136-140 */
double orc_pt_dist(const double* ctrl /*[N][3]*/, int32_t n_pts);

/* CPU twin of the device-side batched optimiser loop (fuelgpu_bspline_optimize_batch):
 * NOT a restatement of NLopt (third-party, absent; SURVEY 8c).  It restates the parts of
 * BsplineOptimizer::optimize() that are in-tree -- clamp to box +-0.1 (:175-200), bounds
 * (:202-217), best-x tracking (costFunction :693-706), maxeval stop -- around a
 * projected L-BFGS.  Used to check the device loop iterate-for-iterate and as the timed
 * CPU baseline for the trajectory batch. */
typedef struct {
  int32_t max_eval;   /* max_iteration_num_[id] */
  int32_t lbfgs_m;    /* history length */
  double xtol_rel;    /* 1e-5, :173 */
  int32_t flags;      /* ORC_SOLVE_* (same bits as FUELGPU_SOLVE_*) */
  int32_t reserved;
} OrcSolveParams;
/* FUELGPU_SOLVE_EXACT_EVALS: a vanished projected gradient re-evaluates in place until max_eval, a failed line
 * search drops the history and goes on from steepest descent, and there is no xtol stop */
#define ORC_SOLVE_EXACT_EVALS 1
void orc_optimize_batch(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                        const OrcTrajConst* tc, int32_t n_pts, int32_t cost_mask, int32_t B,
                        const OrcSolveParams* sp, double* x /*[B][nvar] in/out*/,
                        double* f_best /*[B]*/, int32_t* n_eval /*[B]*/, int threads);

/* What the solver decided for one trajectory: event counts, and when the first of the two rare events happened
 * (the evaluation count at that moment; -1: never). */
typedef struct {
  int32_t n_kept;          /* (s, y) pairs stored */
  int32_t n_curv_reject;   /* pairs refused by the curvature test */
  int32_t n_full_reject;   /* ... of them while the history ring was full */
  int32_t n_restart;       /* non-descent directions replaced by steepest descent */
  int32_t n_ls_fail;       /* line searches that ended without an Armijo step */
  int32_t first_full_reject;
  int32_t first_ls_fail;
} OrcSolveTrace;
/* orc_optimize_batch with a decision trace (either output may be NULL; results are bit for bit those of
 * orc_optimize_batch).  margin [B][max_eval]: entry k-1 is the smallest relative margin of every branch decision
 * taken while the evaluation count was <= k -- pgn2 > 1e-24, g.d < 0, f < best, the Armijo test, the curvature
 * test and the xtol test -- so a solver that rounds differently takes the same path through its first k
 * evaluations whenever its disagreement stays below that margin. */
void orc_optimize_batch_traced(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                               const OrcTrajConst* tc, int32_t n_pts, int32_t cost_mask, int32_t B,
                               const OrcSolveParams* sp, double* x, double* f_best, int32_t* n_eval,
                               OrcSolveTrace* trace /*[B]*/, double* margin /*[B][max_eval]*/, int threads);

#ifdef __cplusplus
}
#endif
#endif
