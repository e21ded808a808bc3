/*
 * fuel_oracle.c -- CPU restatement of FUEL's per-replan hot path (see fuel_oracle.h).
 *
 * TEST INFRASTRUCTURE ONLY -- never linked into, imported by or called from the product
 * (fuel_b200/).  PARITY UNPINNED by reference tests (the reference has none for this
 * path); pinned against brute force / scipy / finite differences in tests/.
 *
 * Citations are file:line under /root/reference/fuel_planner/.
 */
#define _GNU_SOURCE
#include "fuel_oracle.h"

#include <assert.h>
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ------------------------------------------------------------------------------------ */
/* index helpers: plan_env/include/plan_env/sdf_map.h:127-192                           */
/* ------------------------------------------------------------------------------------ */

static inline double res_inv(const OrcGrid* g) { return 1 / g->res; } /* sdf_map.cpp:33 */

/* sdf_map.h:127-130 */
void orc_pos_to_index(const OrcGrid* g, const double pos[3], int32_t id[3]) {
  const double ri = res_inv(g);
  for (int i = 0; i < 3; ++i) id[i] = (int32_t)floor((pos[i] - g->origin[i]) * ri);
}

/* sdf_map.h:132-135 */
void orc_index_to_pos(const OrcGrid* g, const int32_t id[3], double pos[3]) {
  for (int i = 0; i < 3; ++i) pos[i] = (id[i] + 0.5) * g->res + g->origin[i];
}

/* sdf_map.h:145-147 */
static inline int64_t to_address(const OrcGrid* g, int x, int y, int z) {
  return (int64_t)x * g->n[1] * g->n[2] + (int64_t)y * g->n[2] + z;
}

/* map_max_boundary_ = origin + map_size_, sdf_map.cpp:34-39.  map_size_ here is n*res
 * (the reference derives n = ceil(size/res) from size; fixtures give n and res). */
static inline double map_max(const OrcGrid* g, int i) {
  return g->origin[i] + (g->map_size[i] > 0.0 ? g->map_size[i] : g->n[i] * g->res);
}

/* sdf_map.h:153-161 */
int orc_is_in_map_pos(const OrcGrid* g, const double pos[3]) {
  if (pos[0] < g->origin[0] + 1e-4 || pos[1] < g->origin[1] + 1e-4 || pos[2] < g->origin[2] + 1e-4)
    return 0;
  if (pos[0] > map_max(g, 0) - 1e-4 || pos[1] > map_max(g, 1) - 1e-4 ||
      pos[2] > map_max(g, 2) - 1e-4)
    return 0;
  return 1;
}

/* sdf_map.h:163-169 */
static inline int is_in_map_idx(const OrcGrid* g, const int32_t id[3]) {
  if (id[0] < 0 || id[1] < 0 || id[2] < 0) return 0;
  if (id[0] > g->n[0] - 1 || id[1] > g->n[1] - 1 || id[2] > g->n[2] - 1) return 0;
  return 1;
}

/* sdf_map.h:171-178; box_min_/box_max_ = posToIndex(box_mind_/box_maxd_), sdf_map.cpp:83-84 */
static inline int is_in_box_idx(const OrcGrid* g, const int32_t bmin[3], const int32_t bmax[3],
                                const int32_t id[3]) {
  (void)g;
  for (int i = 0; i < 3; ++i)
    if (id[i] < bmin[i] || id[i] >= bmax[i]) return 0;
  return 1;
}

/* sdf_map.h:194-200: occ < clamp_min_log-1e-3 -> UNKNOWN; occ > min_occupancy_log -> OCCUPIED */
void orc_tristate_from_logodds(const double* logodds, int64_t n, double clamp_min_log,
                               double min_occupancy_log, uint8_t* tri) {
  for (int64_t i = 0; i < n; ++i) {
    double occ = logodds[i];
    if (occ < clamp_min_log - 1e-3)
      tri[i] = ORC_UNKNOWN;
    else if (occ > min_occupancy_log)
      tri[i] = ORC_OCCUPIED;
    else
      tri[i] = ORC_FREE;
  }
}

/* getOccupancy(idx), sdf_map.h:194-200: -1 when out of map */
static inline int get_occupancy(const OrcGrid* g, const uint8_t* tri, const int32_t id[3]) {
  if (!is_in_map_idx(g, id)) return -1;
  return (int)tri[to_address(g, id[0], id[1], id[2])];
}

/* ------------------------------------------------------------------------------------ */
/* ESDF: plan_env/src/sdf_map.cpp:116-241                                                */
/* ------------------------------------------------------------------------------------ */

/* fillESDF, sdf_map.cpp:116-150.  f[] holds f_get_val(q) for q in [start,end] (indexed by
 * q, so the `start`-offset indexing of v[]/z[] is the reference's); out[q] receives
 * f_set_val(q, val).  v/z are the VLAs of :117-118. */
static void fill_esdf(const double* f, double* out, int start, int end, int* v, double* z) {
  int k = start;
  v[start] = start;
  z[start] = -DBL_MAX;
  z[start + 1] = DBL_MAX;

  for (int q = start + 1; q <= end; q++) {
    k++;
    double s;
    do {
      k--;
      s = ((f[q] + q * q) - (f[v[k]] + v[k] * v[k])) / (2 * q - 2 * v[k]);
    } while (s <= z[k]);
    k++;
    v[k] = q;
    z[k] = s;
    z[k + 1] = DBL_MAX;
  }

  k = start;
  for (int q = start; q <= end; q++) {
    while (z[k + 1] < q) k++;
    double val = (q - v[k]) * (q - v[k]) + f[v[k]];
    out[q] = val;
  }
}

/* one 3-pass transform, sdf_map.cpp:156-199 (and :201-231 for the negative field).
 * site(adr) selects the pass-z seed.  mode: 0 optimistic (:156-166), 1 non-optimistic
 * (:167-181), 2 negative field (:203-214). */
static void esdf_three_pass(const OrcGrid* g, const int8_t* inflate, const uint8_t* tri,
                            const int32_t bmin[3], const int32_t bmax[3], int mode, double* out,
                            double* tmp1, double* tmp2, int threads) {
  const int nmax = (g->n[0] > g->n[1] ? (g->n[0] > g->n[2] ? g->n[0] : g->n[2])
                                      : (g->n[1] > g->n[2] ? g->n[1] : g->n[2]));
  (void)threads;
#pragma omp parallel num_threads(threads)
  {
    double* f = (double*)malloc(sizeof(double) * (nmax + 2));
    double* o = (double*)malloc(sizeof(double) * (nmax + 2));
    int* v = (int*)malloc(sizeof(int) * (nmax + 2));
    double* z = (double*)malloc(sizeof(double) * (nmax + 2));

    /* pass along z, sdf_map.cpp:156-181 / :203-214 */
#pragma omp for collapse(2) schedule(static)
    for (int x = bmin[0]; x <= bmax[0]; x++)
      for (int y = bmin[1]; y <= bmax[1]; y++) {
        for (int zz = bmin[2]; zz <= bmax[2]; zz++) {
          int64_t adr = to_address(g, x, y, zz);
          int site;
          if (mode == 0)
            site = inflate[adr] == 1;
          else if (mode == 1)
            site = (inflate[adr] == 1 || tri[adr] == ORC_UNKNOWN);
          else
            site = inflate[adr] == 0;
          f[zz] = site ? 0 : DBL_MAX;
        }
        fill_esdf(f, o, bmin[2], bmax[2], v, z);
        for (int zz = bmin[2]; zz <= bmax[2]; zz++) tmp1[to_address(g, x, y, zz)] = o[zz];
      }

    /* pass along y, sdf_map.cpp:183-190 */
#pragma omp for collapse(2) schedule(static)
    for (int x = bmin[0]; x <= bmax[0]; x++)
      for (int zz = bmin[2]; zz <= bmax[2]; zz++) {
        for (int y = bmin[1]; y <= bmax[1]; y++) f[y] = tmp1[to_address(g, x, y, zz)];
        fill_esdf(f, o, bmin[1], bmax[1], v, z);
        for (int y = bmin[1]; y <= bmax[1]; y++) tmp2[to_address(g, x, y, zz)] = o[y];
      }

    /* pass along x, sdf_map.cpp:191-199: distance = resolution_ * sqrt(val) */
#pragma omp for collapse(2) schedule(static)
    for (int y = bmin[1]; y <= bmax[1]; y++)
      for (int zz = bmin[2]; zz <= bmax[2]; zz++) {
        for (int x = bmin[0]; x <= bmax[0]; x++) f[x] = tmp2[to_address(g, x, y, zz)];
        fill_esdf(f, o, bmin[0], bmax[0], v, z);
        for (int x = bmin[0]; x <= bmax[0]; x++) out[to_address(g, x, y, zz)] = g->res * sqrt(o[x]);
      }

    free(f);
    free(o);
    free(v);
    free(z);
  }
}

/* updateESDF3d, sdf_map.cpp:152-241 */
void orc_update_esdf3d(const OrcGrid* g, const int8_t* inflate, const uint8_t* tri,
                       const int32_t bmin[3], const int32_t bmax[3], int optimistic,
                       int signed_dist, double* dist, double* dist_neg, double* tmp1,
                       double* tmp2, int threads) {
  if (threads < 1) threads = 1;
  esdf_three_pass(g, inflate, tri, bmin, bmax, optimistic ? 0 : 1, dist, tmp1, tmp2, threads);
  if (signed_dist) {
    esdf_three_pass(g, inflate, tri, bmin, bmax, 2, dist_neg, tmp1, tmp2, threads);
    /* merge, sdf_map.cpp:232-239 */
    for (int x = bmin[0]; x <= bmax[0]; ++x)
      for (int y = bmin[1]; y <= bmax[1]; ++y)
        for (int z = bmin[2]; z <= bmax[2]; ++z) {
          int64_t idx = to_address(g, x, y, z);
          if (dist_neg[idx] > 0.0) dist[idx] += (-dist_neg[idx] + g->res);
        }
  }
}

/* clearAndInflateLocalMap, sdf_map.cpp:364-472 */
void orc_clear_and_inflate(const OrcGrid* g, uint8_t* tri, int8_t* inflate, const int32_t bmin[3],
                           const int32_t bmax[3], int inf_step, int ceil_id) {
  const int64_t nvox = (int64_t)g->n[0] * g->n[1] * g->n[2];
  /* clean outdated occupancy, :440-444 */
  for (int x = bmin[0]; x <= bmax[0]; ++x)
    for (int y = bmin[1]; y <= bmax[1]; ++y)
      for (int z = bmin[2]; z <= bmax[2]; ++z) inflate[to_address(g, x, y, z)] = 0;
  /* inflate newest occupied cells, :447-460; inflatePoint "all inflate", sdf_map.h:257-264 */
  for (int x = bmin[0]; x <= bmax[0]; ++x)
    for (int y = bmin[1]; y <= bmax[1]; ++y)
      for (int z = bmin[2]; z <= bmax[2]; ++z) {
        if (tri[to_address(g, x, y, z)] == ORC_OCCUPIED) { /* occupancy_buffer_ > min_occupancy_log_ */
          for (int dx = -inf_step; dx <= inf_step; ++dx)
            for (int dy = -inf_step; dy <= inf_step; ++dy)
              for (int dz = -inf_step; dz <= inf_step; ++dz) {
                /* toAddress on the raw (possibly out-of-range) index, checked only as a linear
                 * address: :452-458 */
                const int64_t idx_inf = to_address(g, x + dx, y + dy, z + dz);
                if (idx_inf >= 0 && idx_inf < nvox) inflate[idx_inf] = 1;
              }
        }
      }
  /* virtual ceiling, :462-470: occupancy_buffer_ = clamp_max_log_ (-> OCCUPIED) */
  if (ceil_id >= 0 && ceil_id < g->n[2])
    for (int x = bmin[0]; x <= bmax[0]; ++x)
      for (int y = bmin[1]; y <= bmax[1]; ++y) tri[to_address(g, x, y, ceil_id)] = ORC_OCCUPIED;
}

/* getDistance(idx), sdf_map.h:228-231 */
static inline double get_distance(const OrcGrid* g, const double* dist_buf, const int32_t id[3]) {
  if (!is_in_map_idx(g, id)) return -1;
  return dist_buf[to_address(g, id[0], id[1], id[2])];
}

/* getDistWithGrad, sdf_map.cpp:497-536 */
double orc_dist_with_grad(const OrcGrid* g, const double* dist_buf, const double pos[3],
                          double grad[3]) {
  if (!orc_is_in_map_pos(g, pos)) {
    grad[0] = grad[1] = grad[2] = 0;
    return 0;
  }
  const double ri = res_inv(g);
  double pos_m[3], idx_pos[3], diff[3];
  int32_t idx[3];
  for (int i = 0; i < 3; ++i) pos_m[i] = pos[i] - 0.5 * g->res * 1.0;
  orc_pos_to_index(g, pos_m, idx);
  orc_index_to_pos(g, idx, idx_pos);
  for (int i = 0; i < 3; ++i) diff[i] = (pos[i] - idx_pos[i]) * ri;

  double values[2][2][2];
  for (int x = 0; x < 2; x++)
    for (int y = 0; y < 2; y++)
      for (int z = 0; z < 2; z++) {
        int32_t cur[3] = { idx[0] + x, idx[1] + y, idx[2] + z };
        values[x][y][z] = get_distance(g, dist_buf, cur);
      }

  double v00 = (1 - diff[0]) * values[0][0][0] + diff[0] * values[1][0][0];
  double v01 = (1 - diff[0]) * values[0][0][1] + diff[0] * values[1][0][1];
  double v10 = (1 - diff[0]) * values[0][1][0] + diff[0] * values[1][1][0];
  double v11 = (1 - diff[0]) * values[0][1][1] + diff[0] * values[1][1][1];
  double v0 = (1 - diff[1]) * v00 + diff[1] * v10;
  double v1 = (1 - diff[1]) * v01 + diff[1] * v11;
  double dist = (1 - diff[2]) * v0 + diff[2] * v1;

  grad[2] = (v1 - v0) * ri;
  grad[1] = ((1 - diff[2]) * (v10 - v00) + diff[2] * (v11 - v01)) * ri;
  grad[0] = (1 - diff[2]) * (1 - diff[1]) * (values[1][0][0] - values[0][0][0]);
  grad[0] += (1 - diff[2]) * diff[1] * (values[1][1][0] - values[0][1][0]);
  grad[0] += diff[2] * (1 - diff[1]) * (values[1][0][1] - values[0][0][1]);
  grad[0] += diff[2] * diff[1] * (values[1][1][1] - values[0][1][1]);
  grad[0] *= ri;
  return dist;
}

void orc_dist_with_grad_batch(const OrcGrid* g, const double* dist_buf, int64_t n,
                              const double* pos, double* dist, double* grad) {
  for (int64_t i = 0; i < n; ++i) dist[i] = orc_dist_with_grad(g, dist_buf, pos + 3 * i, grad + 3 * i);
}

/* ------------------------------------------------------------------------------------ */
/* Frontier: active_perception/src/frontier_finder.cpp                                   */
/* ------------------------------------------------------------------------------------ */

typedef struct {
  double* cells; /* n*3 positions, as Frontier::cells_ (frontier_finder.h:38) */
  int32_t* addr; /* n addresses (toAddress of posToIndex(cell)) */
  int32_t n, cap;
  double* filtered; /* m*3, Frontier::filtered_cells_ */
  int32_t m;
  double average[3], box_min[3], box_max[3];
} Ftr;

struct OrcFrontierResult {
  Ftr* f;
  int32_t n, cap;
};

static void ftr_init(Ftr* f) { memset(f, 0, sizeof(*f)); }
static void ftr_free(Ftr* f) {
  free(f->cells);
  free(f->addr);
  free(f->filtered);
}
static void ftr_push(Ftr* f, const double pos[3], int32_t addr) {
  if (f->n == f->cap) {
    f->cap = f->cap ? f->cap * 2 : 256;
    f->cells = (double*)realloc(f->cells, sizeof(double) * 3 * f->cap);
    f->addr = (int32_t*)realloc(f->addr, sizeof(int32_t) * f->cap);
  }
  memcpy(f->cells + 3 * f->n, pos, sizeof(double) * 3);
  f->addr[f->n] = addr;
  f->n++;
}
static void res_push(OrcFrontierResult* r, Ftr* f) { /* moves f */
  if (r->n == r->cap) {
    r->cap = r->cap ? r->cap * 2 : 16;
    r->f = (Ftr*)realloc(r->f, sizeof(Ftr) * r->cap);
  }
  r->f[r->n++] = *f;
}

typedef struct {
  const OrcGrid* g;
  const uint8_t* tri;
  int8_t* flag;
  int32_t box_min[3], box_max[3]; /* mp_->box_min_/box_max_ */
  const OrcFrontierParams* p;
} FCtx;

/* knownfree, frontier_finder.cpp:875-877 */
static inline int knownfree(const FCtx* c, const int32_t id[3]) {
  return get_occupancy(c->g, c->tri, id) == ORC_FREE;
}

/* isNeighborUnknown + sixNeighbors, frontier_finder.cpp:862-869, :811-829 */
static inline int is_neighbor_unknown(const FCtx* c, const int32_t v[3]) {
  static const int d6[6][3] = { { -1, 0, 0 }, { 1, 0, 0 }, { 0, -1, 0 },
                                { 0, 1, 0 },  { 0, 0, -1 }, { 0, 0, 1 } };
  for (int i = 0; i < 6; ++i) {
    int32_t nb[3] = { v[0] + d6[i][0], v[1] + d6[i][1], v[2] + d6[i][2] };
    if (get_occupancy(c->g, c->tri, nb) == ORC_UNKNOWN) return 1;
  }
  return 0;
}

int orc_is_frontier_cell(const OrcGrid* g, const uint8_t* tri, const int32_t id[3]) {
  FCtx c;
  memset(&c, 0, sizeof(c));
  c.g = g;
  c.tri = tri;
  return knownfree(&c, id) && is_neighbor_unknown(&c, id);
}

/* isFrontierChanged, frontier_finder.cpp:365-372 */
int orc_frontier_is_changed(const OrcGrid* g, const uint8_t* tri, const int32_t* addr, int32_t n) {
  const int64_t nyz = (int64_t)g->n[1] * g->n[2];
  for (int32_t i = 0; i < n; ++i) {
    int32_t id[3] = { (int32_t)(addr[i] / nyz), (int32_t)((addr[i] % nyz) / g->n[2]),
                      (int32_t)(addr[i] % g->n[2]) };
    if (!orc_is_frontier_cell(g, tri, id)) return 1;
  }
  return 0;
}

/* --- PCL VoxelGrid<PointXYZ>::applyFilter restated (PCL 1.8 voxel_grid.hpp; third party,
 * not under /root/reference; UNPINNED).  Called at frontier_finder.cpp:757-774.
 *   - points cast to float32 (:762 emplace_back(cell[0],cell[1],cell[2]) into PointXYZ)
 *   - leaf_size (double res*down_sample) narrowed to float by setLeafSize(float,float,float)
 *   - inverse_leaf_size = 1.0f / leaf_size
 *   - min_b = floor(min_p * inv), div_b = max_b - min_b + 1
 *   - leaf index = ijk0 + ijk1*div_b0 + ijk2*div_b0*div_b1,
 *       ijk = (int)(floorf(p*inv) - (float)min_b)
 *   - points sorted by leaf index; centroid = float sum / float count, emitted in ascending
 *     leaf index.  Within-leaf accumulation order: ascending original index (std::sort is
 *     not stable in PCL; this is the documented convention, SURVEY 8c).                 */
typedef struct {
  int32_t leaf;
  int32_t idx;
} LeafIdx;
static int leaf_cmp(const void* a, const void* b) {
  const LeafIdx* x = (const LeafIdx*)a;
  const LeafIdx* y = (const LeafIdx*)b;
  if (x->leaf != y->leaf) return x->leaf < y->leaf ? -1 : 1;
  return x->idx < y->idx ? -1 : (x->idx > y->idx ? 1 : 0);
}

/* The filter itself on float32 points (what a pcl::PointCloud<pcl::PointXYZ> holds); out has room for n points.
 * Exported because oracle/ref_standin/pcl/filters/voxel_grid.h -- the stand-in the reference's frontier_finder.cpp is
 * compiled against for oracle/_ref -- must run the SAME reconstruction (PCL is third party and absent). */
int32_t orc_voxelgrid_f32(const float* pf, int32_t n, float leaf, float* out) {
  const float inv = 1.0f / leaf;
  float minp[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, maxp[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  for (int32_t i = 0; i < n; ++i)
    for (int k = 0; k < 3; ++k) {
      const float v = pf[3 * i + k];
      if (v < minp[k]) minp[k] = v;
      if (v > maxp[k]) maxp[k] = v;
    }
  int32_t min_b[3], max_b[3], div_b[3];
  for (int k = 0; k < 3; ++k) {
    min_b[k] = (int32_t)floorf(minp[k] * inv);
    max_b[k] = (int32_t)floorf(maxp[k] * inv);
    div_b[k] = max_b[k] - min_b[k] + 1;
  }
  LeafIdx* li = (LeafIdx*)malloc(sizeof(LeafIdx) * (n > 0 ? n : 1));
  for (int32_t i = 0; i < n; ++i) {
    int32_t ijk[3];
    for (int k = 0; k < 3; ++k)
      ijk[k] = (int32_t)(floorf(pf[3 * i + k] * inv) - (float)min_b[k]);
    li[i].leaf = ijk[0] + ijk[1] * div_b[0] + ijk[2] * div_b[0] * div_b[1];
    li[i].idx = i;
  }
  qsort(li, n, sizeof(LeafIdx), leaf_cmp);
  int32_t cnt = 0;
  int32_t i = 0;
  while (i < n) {
    int32_t j = i;
    float s[3] = { 0.f, 0.f, 0.f };
    while (j < n && li[j].leaf == li[i].leaf) {
      for (int k = 0; k < 3; ++k) s[k] += pf[3 * li[j].idx + k];
      ++j;
    }
    const float fc = (float)(j - i);
    for (int k = 0; k < 3; ++k) out[3 * cnt + k] = s[k] / fc;
    ++cnt;
    i = j;
  }
  free(li);
  return cnt;
}

static void downsample(const FCtx* c, const double* cells, int32_t n, double** out, int32_t* m) {
  const double leaf_size_d = c->g->res * c->p->down_sample; /* frontier_finder.cpp:765 */
  const float leaf = (float)leaf_size_d;
  float* pf = (float*)malloc(sizeof(float) * 3 * (n > 0 ? n : 1));
  float* of = (float*)malloc(sizeof(float) * 3 * (n > 0 ? n : 1));
  for (int32_t i = 0; i < 3 * n; ++i) pf[i] = (float)cells[i];
  const int32_t cnt = orc_voxelgrid_f32(pf, n, leaf, of);
  double* o = (double*)malloc(sizeof(double) * 3 * (n > 0 ? n : 1));
  for (int32_t i = 0; i < 3 * cnt; ++i) o[i] = (double)of[i]; /* :772-773 float->double */
  free(pf);
  free(of);
  *out = o;
  *m = cnt;
}

/* computeFrontierInfo, frontier_finder.cpp:374-390 */
static void compute_frontier_info(const FCtx* c, Ftr* f) {
  f->average[0] = f->average[1] = f->average[2] = 0;
  for (int k = 0; k < 3; ++k) f->box_max[k] = f->box_min[k] = f->cells[k];
  for (int32_t i = 0; i < f->n; ++i) {
    for (int k = 0; k < 3; ++k) {
      double v = f->cells[3 * i + k];
      f->average[k] += v;
      f->box_min[k] = f->box_min[k] < v ? f->box_min[k] : v;
      f->box_max[k] = f->box_max[k] > v ? f->box_max[k] : v;
    }
  }
  for (int k = 0; k < 3; ++k) f->average[k] /= (double)f->n;
  free(f->filtered);
  downsample(c, f->cells, f->n, &f->filtered, &f->m);
}

/* --- Eigen 3.3 EigenSolver<Matrix2d> on a symmetric [[a,b],[b,d]], reconstructed
 * (third party, absent; UNPINNED).  RealSchur::computeFromHessenberg ->
 * findSmallSubdiagEntry / splitOffTwoRows / JacobiRotation::makeGivens, then
 * EigenSolver::doComputeEigenvectors back-substitution, column normalisation.
 * Returns the eigenvector of the larger eigenvalue with Eigen's sign convention;
 * ties pick index 0 (the `values[i] > max_eigenvalue` scan, frontier_finder.cpp:207-212). */
static void make_givens(double p, double q, double* c, double* s) {
  if (q == 0.0) {
    *c = p < 0 ? -1.0 : 1.0;
    *s = 0.0;
  } else if (p == 0.0) {
    *c = 0.0;
    *s = q < 0 ? 1.0 : -1.0;
  } else if (fabs(p) > fabs(q)) {
    double t = q / p;
    double u = sqrt(1.0 + t * t);
    if (p < 0) u = -u;
    *c = 1.0 / u;
    *s = -t * (*c);
  } else {
    double t = p / q;
    double u = sqrt(1.0 + t * t);
    if (q < 0) u = -u;
    *s = -1.0 / u;
    *c = -t * (*s);
  }
}

/* eigenvalues().real() and eigenvectors().real() of EigenSolver<Matrix2d> on [[a,b],[b,d]] under the reconstructed
 * Eigen 3.3 convention: vals[i], vecs[row][col] (column i = eigenvector i).  Exported for
 * oracle/ref_standin/Eigen/Eigenvalues (see orc_voxelgrid_f32). */
void orc_eigen_sym2x2(double a, double b, double d, double vals_out[2], double vecs_out[2][2]) {
  /* T starts as the matrix itself (Hessenberg reduction of a 2x2 is the identity) */
  double T[2][2] = { { a, b }, { b, d } };
  double U[2][2] = { { 1, 0 }, { 0, 1 } };
  /* norm used by RealSchur as the scale for zero tests: sum of |T(i,j)| over the
   * upper-Hessenberg part */
  double norm = fabs(a) + fabs(b) + fabs(b) + fabs(d);
  if (norm != 0.0) {
    double s = fabs(T[0][0]) + fabs(T[1][1]);
    double thr = s * DBL_EPSILON;
    if (!(fabs(T[1][0]) <= thr)) {
      /* splitOffTwoRows */
      double p = 0.5 * (T[0][0] - T[1][1]);
      double q = p * p + T[1][0] * T[0][1];
      if (q >= 0) {
        double z = sqrt(fabs(q));
        double c, sn;
        if (p >= 0)
          make_givens(p + z, T[1][0], &c, &sn);
        else
          make_givens(p - z, T[1][0], &c, &sn);
        /* applyOnTheLeft(0,1,rot.adjoint()): rows x=row0,y=row1 with J^T:
         *   x' = c*x - s*y ; y' = s*x + c*y   (adjoint of [[c,s],[-s,c]]) */
        for (int j = 0; j < 2; ++j) {
          double x = T[0][j], y = T[1][j];
          T[0][j] = c * x - sn * y;
          T[1][j] = sn * x + c * y;
        }
        /* applyOnTheRight(0,1,rot): cols x=col0,y=col1: x' = c*x - s*y ; y' = s*x + c*y */
        for (int i = 0; i < 2; ++i) {
          double x = T[i][0], y = T[i][1];
          T[i][0] = c * x - sn * y;
          T[i][1] = sn * x + c * y;
        }
        T[1][0] = 0.0;
        for (int i = 0; i < 2; ++i) {
          double x = U[i][0], y = U[i][1];
          U[i][0] = c * x - sn * y;
          U[i][1] = sn * x + c * y;
        }
      }
    } else {
      T[1][0] = 0.0;
    }
  }
  /* doComputeEigenvectors: back-substitute on upper-triangular T.
   * vec0 (Schur basis) = (1,0); vec1 = (-T01/(T00-T11), 1) */
  double e0[2] = { 1.0, 0.0 };
  double e1[2];
  {
    double w = T[0][0] - T[1][1];
    double r = T[0][1];
    if (w != 0.0)
      e1[0] = -r / w;
    else
      e1[0] = -r / (DBL_EPSILON * norm);
    e1[1] = 1.0;
    /* overflow control in Eigen rescales only when huge; irrelevant here */
  }
  double v0[2] = { U[0][0] * e0[0] + U[0][1] * e0[1], U[1][0] * e0[0] + U[1][1] * e0[1] };
  double v1[2] = { U[0][0] * e1[0] + U[0][1] * e1[1], U[1][0] * e1[0] + U[1][1] * e1[1] };
  double n0 = sqrt(v0[0] * v0[0] + v0[1] * v0[1]);
  double n1 = sqrt(v1[0] * v1[0] + v1[1] * v1[1]);
  if (n0 > 0) { v0[0] /= n0; v0[1] /= n0; }
  if (n1 > 0) { v1[0] /= n1; v1[1] /= n1; }
  vals_out[0] = T[0][0], vals_out[1] = T[1][1];
  vecs_out[0][0] = v0[0], vecs_out[1][0] = v0[1];
  vecs_out[0][1] = v1[0], vecs_out[1][1] = v1[1];
}

void orc_principal_axis_2x2(double a, double b, double d, double pc[2]) {
  double vals[2], vecs[2][2];
  orc_eigen_sym2x2(a, b, d, vals, vecs);
  /* pick the larger eigenvalue, ties -> index 0 (frontier_finder.cpp:205-212) */
  int max_idx = 0;
  double max_ev = -1000000;
  for (int i = 0; i < 2; ++i)
    if (vals[i] > max_ev) {
      max_idx = i;
      max_ev = vals[i];
    }
  pc[0] = vecs[0][max_idx];
  pc[1] = vecs[1][max_idx];
}

/* splitHorizontally, frontier_finder.cpp:179-242.  Returns 1 and appends the pieces
 * to `splits` (in ftr1-subtree, ftr2-subtree order) if the frontier was split. */
static int split_horizontally(const FCtx* c, const Ftr* fr, OrcFrontierResult* splits) {
  const double mean[2] = { fr->average[0], fr->average[1] };
  int need_split = 0;
  for (int32_t i = 0; i < fr->m; ++i) {
    double dx = fr->filtered[3 * i] - mean[0], dy = fr->filtered[3 * i + 1] - mean[1];
    if (sqrt(dx * dx + dy * dy) > c->p->cluster_size_xy) { /* Vector2d::norm() */
      need_split = 1;
      break;
    }
  }
  if (!need_split) return 0;

  /* covariance of filtered cells, :194-200 */
  double cov[2][2] = { { 0, 0 }, { 0, 0 } };
  for (int32_t i = 0; i < fr->m; ++i) {
    double dx = fr->filtered[3 * i] - mean[0], dy = fr->filtered[3 * i + 1] - mean[1];
    cov[0][0] += dx * dx;
    cov[0][1] += dx * dy;
    cov[1][0] += dy * dx;
    cov[1][1] += dy * dy;
  }
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 2; ++j) cov[i][j] /= (double)fr->m;

  double pc[2];
  orc_principal_axis_2x2(cov[0][0], cov[1][0], cov[1][1], pc);

  /* partition ALL cells by sign of projection, :216-224 */
  Ftr f1, f2;
  ftr_init(&f1);
  ftr_init(&f2);
  for (int32_t i = 0; i < fr->n; ++i) {
    double dx = fr->cells[3 * i] - mean[0], dy = fr->cells[3 * i + 1] - mean[1];
    if (dx * pc[0] + dy * pc[1] >= 0)
      ftr_push(&f1, fr->cells + 3 * i, fr->addr[i]);
    else
      ftr_push(&f2, fr->cells + 3 * i, fr->addr[i]);
  }
  /* A one-sided partition would recurse forever in the reference (computeFrontierInfo
   * on an empty cells_ is UB at :377).  Cannot happen when need_split holds and the mean
   * lies inside the hull; guard so the oracle terminates instead of crashing. */
  if (f1.n == 0 || f2.n == 0) {
    ftr_free(&f1);
    ftr_free(&f2);
    return 0;
  }
  compute_frontier_info(c, &f1);
  compute_frontier_info(c, &f2);

  /* recurse, :229-239 */
  if (!split_horizontally(c, &f1, splits))
    res_push(splits, &f1);
  else
    ftr_free(&f1);
  if (!split_horizontally(c, &f2, splits))
    res_push(splits, &f2);
  else
    ftr_free(&f2);
  return 1;
}

static int addr_cmp_perm(const void* a, const void* b, void* arg) {
  const int32_t* addr = (const int32_t*)arg;
  int32_t x = addr[*(const int32_t*)a], y = addr[*(const int32_t*)b];
  return x < y ? -1 : (x > y ? 1 : 0);
}

/* expandFrontier, frontier_finder.cpp:123-164 */
static void expand_frontier(const FCtx* c, const int32_t first[3], OrcFrontierResult* tmp) {
  const OrcGrid* g = c->g;
  Ftr ex;
  ftr_init(&ex);
  int32_t qcap = 1024, qh = 0, qt = 0;
  int32_t* queue = (int32_t*)malloc(sizeof(int32_t) * 3 * qcap);
  double pos[3];

  orc_index_to_pos(g, first, pos);
  ftr_push(&ex, pos, (int32_t)to_address(g, first[0], first[1], first[2]));
  memcpy(queue + 3 * qt, first, sizeof(int32_t) * 3);
  qt++;
  c->flag[to_address(g, first[0], first[1], first[2])] = 1;

  while (qh < qt) {
    int32_t cur[3] = { queue[3 * qh], queue[3 * qh + 1], queue[3 * qh + 2] };
    qh++;
    /* allNeighbors, :848-860: x outer, y, z inner, centre skipped */
    for (int dx = -1; dx <= 1; ++dx)
      for (int dy = -1; dy <= 1; ++dy)
        for (int dz = -1; dz <= 1; ++dz) {
          if (dx == 0 && dy == 0 && dz == 0) continue;
          int32_t nbr[3] = { cur[0] + dx, cur[1] + dy, cur[2] + dz };
          /* The reference reads frontier_flag_[toadr(nbr)] before isInBox(nbr) (:145-146),
           * which is out-of-bounds UB for nbr outside the map (SURVEY H9).  The box lies
           * inside the map, so an out-of-map nbr is rejected by isInBox anyway: test the
           * map first and never read out of bounds. */
          if (!is_in_map_idx(g, nbr)) continue;
          int64_t adr = to_address(g, nbr[0], nbr[1], nbr[2]);
          if (c->flag[adr] == 1 || !is_in_box_idx(g, c->box_min, c->box_max, nbr) ||
              !(knownfree(c, nbr) && is_neighbor_unknown(c, nbr)))
            continue;
          orc_index_to_pos(g, nbr, pos);
          if (pos[2] < c->p->min_z) continue; /* :152 "Remove noise close to ground" */
          ftr_push(&ex, pos, (int32_t)adr);
          if (qt == qcap) {
            qcap *= 2;
            queue = (int32_t*)realloc(queue, sizeof(int32_t) * 3 * qcap);
          }
          memcpy(queue + 3 * qt, nbr, sizeof(int32_t) * 3);
          qt++;
          c->flag[adr] = 1;
        }
  }
  free(queue);
  if (ex.n > c->p->cluster_min) { /* :157 */
    if (c->p->cell_order == 1) {
      /* canonical order: ascending address (documented deviation knob; the GPU path
       * emits cells in this order, see DESIGN.md "frontier cell order") */
      int32_t* perm = (int32_t*)malloc(sizeof(int32_t) * ex.n);
      for (int32_t i = 0; i < ex.n; ++i) perm[i] = i;
      qsort_r(perm, ex.n, sizeof(int32_t), addr_cmp_perm, ex.addr);
      double* nc = (double*)malloc(sizeof(double) * 3 * ex.n);
      int32_t* na = (int32_t*)malloc(sizeof(int32_t) * ex.n);
      for (int32_t i = 0; i < ex.n; ++i) {
        memcpy(nc + 3 * i, ex.cells + 3 * perm[i], sizeof(double) * 3);
        na[i] = ex.addr[perm[i]];
      }
      free(ex.cells);
      free(ex.addr);
      free(perm);
      ex.cells = nc;
      ex.addr = na;
      ex.cap = ex.n;
    }
    compute_frontier_info(c, &ex);
    res_push(tmp, &ex);
  } else {
    ftr_free(&ex);
  }
}

/* searchFrontiers, frontier_finder.cpp:54-121 (sweep + expand + split) */
OrcFrontierResult* orc_frontier_search(const OrcGrid* g, const uint8_t* tri, int8_t* flag,
                                       const double upd_min[3], const double upd_max[3],
                                       const OrcFrontierParams* p) {
  FCtx c;
  c.g = g;
  c.tri = tri;
  c.flag = flag;
  c.p = p;
  orc_pos_to_index(g, g->box_mind, c.box_min); /* sdf_map.cpp:83-84 */
  orc_pos_to_index(g, g->box_maxd, c.box_max);

  OrcFrontierResult tmp = { 0, 0, 0 };

  /* search box: updated box inflated by (1,1,0.5) and clamped to the exploration box, :94-104 */
  const double infl[3] = { 1, 1, 0.5 };
  double smin[3], smax[3];
  for (int k = 0; k < 3; ++k) {
    smin[k] = upd_min[k] - infl[k];
    smax[k] = upd_max[k] + infl[k];
    smin[k] = smin[k] > g->box_mind[k] ? smin[k] : g->box_mind[k];
    smax[k] = smax[k] < g->box_maxd[k] ? smax[k] : g->box_maxd[k];
  }
  int32_t min_id[3], max_id[3];
  orc_pos_to_index(g, smin, min_id);
  orc_pos_to_index(g, smax, max_id);

  for (int x = min_id[0]; x <= max_id[0]; ++x)
    for (int y = min_id[1]; y <= max_id[1]; ++y)
      for (int z = min_id[2]; z <= max_id[2]; ++z) {
        int32_t cur[3] = { x, y, z };
        /* :113 indexes frontier_flag_ with x == voxel_num when box_maxd_ == map max (UB,
         * SURVEY H9); such a cell is never knownfree, so skipping it is equivalent. */
        if (!is_in_map_idx(g, cur)) continue;
        if (flag[to_address(g, x, y, z)] == 0 && knownfree(&c, cur) && is_neighbor_unknown(&c, cur))
          expand_frontier(&c, cur, &tmp);
      }

  /* splitLargeFrontiers, :166-177 */
  OrcFrontierResult* out = (OrcFrontierResult*)calloc(1, sizeof(OrcFrontierResult));
  for (int32_t i = 0; i < tmp.n; ++i) {
    if (split_horizontally(&c, &tmp.f[i], out))
      ftr_free(&tmp.f[i]);
    else
      res_push(out, &tmp.f[i]);
  }
  free(tmp.f);
  return out;
}

int32_t orc_frontier_count(const OrcFrontierResult* r) { return r->n; }
int32_t orc_frontier_num_cells(const OrcFrontierResult* r, int32_t i) { return r->f[i].n; }
int32_t orc_frontier_num_filtered(const OrcFrontierResult* r, int32_t i) { return r->f[i].m; }
void orc_frontier_get(const OrcFrontierResult* r, int32_t i, int32_t* addr, double* filtered,
                      double avg[3], double bmin[3], double bmax[3]) {
  const Ftr* f = &r->f[i];
  if (addr) memcpy(addr, f->addr, sizeof(int32_t) * f->n);
  if (filtered) memcpy(filtered, f->filtered, sizeof(double) * 3 * f->m);
  for (int k = 0; k < 3; ++k) {
    if (avg) avg[k] = f->average[k];
    if (bmin) bmin[k] = f->box_min[k];
    if (bmax) bmax[k] = f->box_max[k];
  }
}
void orc_frontier_free(OrcFrontierResult* r) {
  if (!r) return;
  for (int32_t i = 0; i < r->n; ++i) ftr_free(&r->f[i]);
  free(r->f);
  free(r);
}

/* ------------------------------------------------------------------------------------ */
/* B-spline cost: bspline_opt/src/bspline_optimizer.cpp                                  */
/* ------------------------------------------------------------------------------------ */

typedef double V3[3];

static inline void v3zero(V3* a, int n) { memset(a, 0, sizeof(V3) * n); }

/* calcSmoothnessCost, :255-282 (gt stays 0: the dt term is commented out at :279-280) */
static void calc_smoothness(const V3* q, int n, double pt_dist, double* cost, V3* gq, double* gt) {
  *cost = 0.0;
  v3zero(gq, n);
  (void)gt;
  for (int i = 0; i < n - 3; i++) {
    double ji[3], tj[3];
    for (int k = 0; k < 3; ++k)
      ji[k] = (q[i + 3][k] - 3 * q[i + 2][k] + 3 * q[i + 1][k] - q[i][k]) / pt_dist;
    *cost += ji[0] * ji[0] + ji[1] * ji[1] + ji[2] * ji[2];
    for (int k = 0; k < 3; ++k) tj[k] = 2 * ji[k] / pt_dist;
    for (int k = 0; k < 3; ++k) {
      gq[i + 0][k] += -tj[k];
      gq[i + 1][k] += 3.0 * tj[k];
      gq[i + 2][k] += -3.0 * tj[k];
      gq[i + 3][k] += tj[k];
    }
  }
}

/* calcDistanceCost, :284-306 (static environment: dynamic_ == false) */
static void calc_distance(const OrcGrid* g, const double* dist_buf, const V3* q, int n,
                          double dist0, double* cost, V3* gq) {
  *cost = 0.0;
  v3zero(gq, n);
  for (int i = 0; i < n; i++) {
    double dg[3];
    double dist = orc_dist_with_grad(g, dist_buf, q[i], dg);
    double nrm = sqrt(dg[0] * dg[0] + dg[1] * dg[1] + dg[2] * dg[2]);
    if (nrm > 1e-4) { /* Vector3d::normalize(): v /= norm() */
      dg[0] /= nrm;
      dg[1] /= nrm;
      dg[2] /= nrm;
    }
    if (dist < dist0) {
      *cost += pow(dist - dist0, 2);
      for (int k = 0; k < 3; ++k) gq[i][k] += 2.0 * (dist - dist0) * dg[k];
    }
  }
}

/* calcFeasibilityCost, :308-353 */
static void calc_feasibility(const V3* q, int n, double dt, double max_vel, double max_acc,
                             int optimize_time, double* cost, V3* gq, double* gt) {
  *cost = 0.0;
  v3zero(gq, n);
  *gt = 0.0;
  const double dt_inv = 1 / dt;
  const double dt_inv2 = dt_inv * dt_inv;
  for (int i = 0; i < n - 1; ++i) {
    for (int k = 0; k < 3; ++k) {
      double vi = (q[i + 1][k] - q[i][k]) * dt_inv;
      double vd = fabs(vi) - max_vel;
      if (vd > 0.0) {
        *cost += pow(vd, 2);
        double sign = vi > 0 ? 1.0 : -1.0;
        double tmp = 2 * vd * sign * dt_inv;
        gq[i][k] += -tmp;
        gq[i + 1][k] += tmp;
        if (optimize_time) *gt += tmp * (-vi);
      }
    }
  }
  for (int i = 0; i < n - 2; ++i) {
    for (int k = 0; k < 3; ++k) {
      double ai = (q[i + 2][k] - 2 * q[i + 1][k] + q[i][k]) * dt_inv2;
      double ad = fabs(ai) - max_acc;
      if (ad > 0.0) {
        *cost += pow(ad, 2);
        double sign = ai > 0 ? 1.0 : -1.0;
        double tmp = 2 * ad * sign * dt_inv2;
        gq[i][k] += tmp;
        gq[i + 1][k] += -2 * tmp;
        gq[i + 2][k] += tmp;
        if (optimize_time) *gt += tmp * ai * (-2) * dt;
      }
    }
  }
}

/* calcStartCost, :355-391 */
static void calc_start(const V3* q, double dt, const double ss[3][3], int optimize_time,
                       double* cost, V3* gq, double* gt) {
  *cost = 0.0;
  for (int i = 0; i < 3; ++i) gq[i][0] = gq[i][1] = gq[i][2] = 0;
  *gt = 0.0;
  const double* q1 = q[0];
  const double* q2 = q[1];
  const double* q3 = q[2];
  double dq[3];
  static const double w_pos = 10.0;
  /* start position */
  for (int k = 0; k < 3; ++k) dq[k] = 1 / 6.0 * (q1[k] + 4 * q2[k] + q3[k]) - ss[0][k];
  *cost += w_pos * (dq[0] * dq[0] + dq[1] * dq[1] + dq[2] * dq[2]);
  for (int k = 0; k < 3; ++k) {
    gq[0][k] += w_pos * 2 * dq[k] * (1 / 6.0);
    gq[1][k] += w_pos * 2 * dq[k] * (4 / 6.0);
    gq[2][k] += w_pos * 2 * dq[k] * (1 / 6.0);
  }
  /* start velocity */
  for (int k = 0; k < 3; ++k) dq[k] = 1 / (2 * dt) * (q3[k] - q1[k]) - ss[1][k];
  *cost += dq[0] * dq[0] + dq[1] * dq[1] + dq[2] * dq[2];
  for (int k = 0; k < 3; ++k) {
    gq[0][k] += 2 * dq[k] * (-1.0) / (2 * dt);
    gq[2][k] += 2 * dq[k] * 1.0 / (2 * dt);
  }
  if (optimize_time) {
    double d = 0;
    for (int k = 0; k < 3; ++k) d += dq[k] * (q3[k] - q1[k]);
    *gt += d / (-dt * dt);
  }
  /* start acceleration */
  for (int k = 0; k < 3; ++k) dq[k] = 1 / (dt * dt) * (q1[k] - 2 * q2[k] + q3[k]) - ss[2][k];
  *cost += dq[0] * dq[0] + dq[1] * dq[1] + dq[2] * dq[2];
  for (int k = 0; k < 3; ++k) {
    gq[0][k] += 2 * dq[k] * 1.0 / (dt * dt);
    gq[1][k] += 2 * dq[k] * (-2.0) / (dt * dt);
    gq[2][k] += 2 * dq[k] * 1.0 / (dt * dt);
  }
  if (optimize_time) {
    double d = 0;
    for (int k = 0; k < 3; ++k) d += dq[k] * (q1[k] - 2 * q2[k] + q3[k]);
    *gt += d / (-dt * dt * dt);
  }
}

/* calcEndCost, :393-431 */
static void calc_end(const V3* q, int n, double dt, const double es[3][3], int n_end,
                     int optimize_time, double* cost, V3* gq, double* gt) {
  *cost = 0.0;
  for (int i = n - 3; i < n; ++i) gq[i][0] = gq[i][1] = gq[i][2] = 0;
  *gt = 0.0;
  const double* q_3 = q[n - 3];
  const double* q_2 = q[n - 2];
  const double* q_1 = q[n - 1];
  double dq[3];
  for (int k = 0; k < 3; ++k) dq[k] = 1 / 6.0 * (q_1[k] + 4 * q_2[k] + q_3[k]) - es[0][k];
  *cost += dq[0] * dq[0] + dq[1] * dq[1] + dq[2] * dq[2];
  for (int k = 0; k < 3; ++k) {
    gq[n - 1][k] += 2 * dq[k] * (1 / 6.0);
    gq[n - 2][k] += 2 * dq[k] * (4 / 6.0);
    gq[n - 3][k] += 2 * dq[k] * (1 / 6.0);
  }
  if (n_end >= 2) {
    for (int k = 0; k < 3; ++k) dq[k] = 1 / (2 * dt) * (q_1[k] - q_3[k]) - es[1][k];
    *cost += dq[0] * dq[0] + dq[1] * dq[1] + dq[2] * dq[2];
    for (int k = 0; k < 3; ++k) {
      gq[n - 1][k] += 2 * dq[k] * 1.0 / (2 * dt);
      gq[n - 3][k] += 2 * dq[k] * (-1.0) / (2 * dt);
    }
    if (optimize_time) {
      double d = 0;
      for (int k = 0; k < 3; ++k) d += dq[k] * (q_1[k] - q_3[k]);
      *gt += d / (-dt * dt);
    }
  }
  if (n_end == 3) {
    for (int k = 0; k < 3; ++k) dq[k] = 1 / (dt * dt) * (q_1[k] - 2 * q_2[k] + q_3[k]) - es[2][k];
    *cost += dq[0] * dq[0] + dq[1] * dq[1] + dq[2] * dq[2];
    for (int k = 0; k < 3; ++k) {
      gq[n - 1][k] += 2 * dq[k] * 1.0 / (dt * dt);
      gq[n - 2][k] += 2 * dq[k] * (-2.0) / (dt * dt);
      gq[n - 3][k] += 2 * dq[k] * 1.0 / (dt * dt);
    }
    if (optimize_time) {
      double d = 0;
      for (int k = 0; k < 3; ++k) d += dq[k] * (q_1[k] - 2 * q_2[k] + q_3[k]);
      *gt += d / (-dt * dt * dt);
    }
  }
}

/* calcWaypointsCost, :433-457 */
static void calc_waypoints(const V3* q, int n, const OrcTrajConst* tc, double* cost, V3* gq) {
  *cost = 0.0;
  v3zero(gq, n);
  for (int i = 0; i < tc->n_waypt; ++i) {
    int idx = tc->waypt_idx[i];
    double dq[3];
    for (int k = 0; k < 3; ++k)
      dq[k] = 1 / 6.0 * (q[idx][k] + 4 * q[idx + 1][k] + q[idx + 2][k]) - tc->waypt[i][k];
    *cost += dq[0] * dq[0] + dq[1] * dq[1] + dq[2] * dq[2];
    for (int k = 0; k < 3; ++k) {
      gq[idx][k] += dq[k] * (2.0 / 6.0);
      gq[idx + 1][k] += dq[k] * (8.0 / 6.0);
      gq[idx + 2][k] += dq[k] * (2.0 / 6.0);
    }
  }
}

/* calcViewCost, :477-502.  Eigen expressions evaluated element-wise in written order: v = dir/sqrt(dir.dir);
 * dn = (q-p) - ((q-p).v) v; g += (2*(I - v vT)) dn; dl = ((q-p).v) v; if |dl| < |dir|: cost += wnl*(|dl|-|dir|)^2,
 * g += ((wnl*2*(|dl|-|dir|)) * v vT) dl / |dl|. */
static void calc_view(const V3* q, int n, const OrcTrajConst* tc, double wnl, double* cost, V3* gq) {
  *cost = 0.0;
  v3zero(gq, n);
  const double* p = tc->view_pt;
  const double* dir = tc->view_dir;
  const double zz = dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2];
  double v[3] = { dir[0], dir[1], dir[2] };
  if (zz > 0) {
    const double nrm = sqrt(zz);
    for (int k = 0; k < 3; ++k) v[k] = dir[k] / nrm;
  }
  double vvT[3][3], I_vvT[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      vvT[i][j] = v[i] * v[j];
      I_vvT[i][j] = (i == j ? 1.0 : 0.0) - vvT[i][j];
    }
  const int i = tc->view_idx;
  const double qp[3] = { q[i][0] - p[0], q[i][1] - p[1], q[i][2] - p[2] };
  const double s = qp[0] * v[0] + qp[1] * v[1] + qp[2] * v[2];
  double dn[3], dl[3];
  for (int k = 0; k < 3; ++k) {
    dl[k] = s * v[k];
    dn[k] = qp[k] - dl[k];
  }
  *cost += dn[0] * dn[0] + dn[1] * dn[1] + dn[2] * dn[2];
  for (int r = 0; r < 3; ++r)
    gq[i][r] += (2 * I_vvT[r][0]) * dn[0] + (2 * I_vvT[r][1]) * dn[1] + (2 * I_vvT[r][2]) * dn[2];
  const double norm_dl = sqrt(dl[0] * dl[0] + dl[1] * dl[1] + dl[2] * dl[2]);
  const double safe_dist = sqrt(zz);
  if (norm_dl < safe_dist) {
    const double e = norm_dl - safe_dist;
    *cost += wnl * (e * e);
    const double c = wnl * 2 * e;
    for (int r = 0; r < 3; ++r)
      gq[i][r] += ((c * vvT[r][0]) * dl[0] + (c * vvT[r][1]) * dl[1] + (c * vvT[r][2]) * dl[2]) / norm_dl;
  }
}

/* calcGuideCost, :462-475 */
static void calc_guide(const V3* q, int n, int order, const OrcTrajConst* tc, double* cost, V3* gq) {
  *cost = 0.0;
  v3zero(gq, n);
  int end_idx = n - order;
  for (int i = order; i < end_idx; i++) {
    const double* gpt = tc->guide[i - order];
    double d[3] = { q[i][0] - gpt[0], q[i][1] - gpt[1], q[i][2] - gpt[2] };
    *cost += d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
    for (int k = 0; k < 3; ++k) gq[i][k] += 2 * d[k];
  }
}

/* calcTimeCost, :504-516 */
static void calc_time(int n, int order, double dt, double time_lb, double* cost, double* gt) {
  double duration = (n - order) * dt;
  *cost = duration;
  *gt = (double)(n - order);
  if (time_lb > 0 && duration < time_lb) {
    static const double w_lb = 10;
    *cost += w_lb * pow(duration - time_lb, 2);
    *gt += w_lb * 2 * (duration - time_lb) * (n - order);
  }
}

double orc_pt_dist(const double* ctrl, int32_t n) { /* :136-140 */
  double d = 0.0;
  for (int i = 0; i < n - 1; ++i) {
    double a = ctrl[3 * (i + 1)] - ctrl[3 * i], b = ctrl[3 * (i + 1) + 1] - ctrl[3 * i + 1],
           c = ctrl[3 * (i + 1) + 2] - ctrl[3 * i + 2];
    d += sqrt(a * a + b * b + c * c);
  }
  return d / (double)n;
}

/* combineCost, :518-647, dim_ == 3.  The two ros::Time::now() calls (:557,:646) are
 * timing instrumentation and are omitted (stated beside every CPU/GPU ratio). */
void orc_combine_cost(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                      const OrcTrajConst* tc, int32_t n, int32_t mask, const double* x,
                      double* f_combine, double* grad) {
  assert(n <= ORC_MAX_PTS);
  V3 q[ORC_MAX_PTS], gt_[ORC_MAX_PTS];
  const int optimize_time = (mask & ORC_MINTIME) != 0; /* :131 */
  const int nvar = optimize_time ? 3 * n + 1 : 3 * n;
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < 3; ++j) q[i][j] = x[3 * i + j];
  const double dt = optimize_time ? x[nvar - 1] : tc->knot_span;

  *f_combine = 0.0;
  for (int i = 0; i < nvar; ++i) grad[i] = 0.0;

  if (mask & ORC_SMOOTHNESS) {
    double f = 0.0, gt = 0.0;
    calc_smoothness((const V3*)q, n, tc->pt_dist, &f, gt_, &gt);
    *f_combine += p->ld_smooth * f;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) grad[3 * i + j] += p->ld_smooth * gt_[i][j];
    if (optimize_time) grad[nvar - 1] += p->ld_smooth * gt;
  }
  if (mask & ORC_DISTANCE) {
    double f = 0.0;
    calc_distance(g, dist_buf, (const V3*)q, n, p->dist0, &f, gt_);
    *f_combine += p->ld_dist * f;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) grad[3 * i + j] += p->ld_dist * gt_[i][j];
  }
  if (mask & ORC_FEASIBILITY) {
    double f = 0.0, gt = 0.0;
    calc_feasibility((const V3*)q, n, dt, p->max_vel, p->max_acc, optimize_time, &f, gt_, &gt);
    *f_combine += p->ld_feasi * f;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) grad[3 * i + j] += p->ld_feasi * gt_[i][j];
    if (optimize_time) grad[nvar - 1] += p->ld_feasi * gt;
  }
  if (mask & ORC_START) {
    double f = 0.0, gt = 0.0;
    calc_start((const V3*)q, dt, tc->start, optimize_time, &f, gt_, &gt);
    *f_combine += p->ld_start * f;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) grad[3 * i + j] += p->ld_start * gt_[i][j];
    if (optimize_time) grad[nvar - 1] += p->ld_start * gt;
  }
  if (mask & ORC_END) {
    double f = 0.0, gt = 0.0;
    calc_end((const V3*)q, n, dt, tc->end, tc->n_end, optimize_time, &f, gt_, &gt);
    *f_combine += p->ld_end * f;
    for (int i = n - 3; i < n; i++)
      for (int j = 0; j < 3; j++) grad[3 * i + j] += p->ld_end * gt_[i][j];
    if (optimize_time) grad[nvar - 1] += p->ld_end * gt;
  }
  if (mask & ORC_GUIDE) {
    double f = 0.0;
    calc_guide((const V3*)q, n, p->order, tc, &f, gt_);
    *f_combine += p->ld_guide * f;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) grad[3 * i + j] += p->ld_guide * gt_[i][j];
  }
  if (mask & ORC_WAYPOINTS) {
    double f = 0.0;
    calc_waypoints((const V3*)q, n, tc, &f, gt_);
    *f_combine += p->ld_waypt * f;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) grad[3 * i + j] += p->ld_waypt * gt_[i][j];
  }
  if (mask & ORC_VIEWCONS) { /* :631-638 */
    double f = 0.0;
    calc_view((const V3*)q, n, tc, p->wnl, &f, gt_);
    *f_combine += p->ld_view * f;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) grad[3 * i + j] += p->ld_view * gt_[i][j];
  }
  if (mask & ORC_MINTIME) {
    double f = 0.0, gt = 0.0;
    calc_time(n, p->order, dt, tc->time_lb, &f, &gt);
    *f_combine += p->ld_time * f;
    grad[nvar - 1] += p->ld_time * gt;
  }
}

void orc_combine_cost_batch(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                            const OrcTrajConst* tc, int32_t n, int32_t mask, int32_t B,
                            const double* x, double* f, double* grad, int threads) {
  const int nvar = (mask & ORC_MINTIME) ? 3 * n + 1 : 3 * n;
  if (threads < 1) threads = 1;
#pragma omp parallel for num_threads(threads) schedule(static)
  for (int b = 0; b < B; ++b)
    orc_combine_cost(g, dist_buf, p, &tc[b], n, mask, x + (int64_t)b * nvar, &f[b],
                     grad + (int64_t)b * nvar);
}

/* ------------------------------------------------------------------------------------ */
/* CPU twin of the device-side batched solver (fuelgpu_bspline_optimize_batch).           */
/* NOT a restatement of NLopt.  Restates what optimize() itself does around the solver   */
/* (bspline_optimizer.cpp:175-217 clamp + bounds, :170 maxeval, :173 xtol_rel, :693-706  */
/* best-x tracking) around the same projected L-BFGS the device runs.                    */
/* ------------------------------------------------------------------------------------ */
#define ORC_MAXM 8
#define ORC_MAXVAR (3 * ORC_MAX_PTS + 1)

static double vdot(const double* a, const double* b, int n) {
  double s = 0.0;
  for (int i = 0; i < n; ++i) s += a[i] * b[i];
  return s;
}

/* relative margin of a decision "a OP b": how far apart the two sides are, over the scale of either */
static double rel_margin(double a, double b, double scale) {
  const double m = fabs(a - b) / scale;
  return m == m ? m : 0.0;  /* NaN (0/0, inf-inf): no margin */
}

static void optimize_one(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                         const OrcTrajConst* tc, int n, int mask, const OrcSolveParams* sp, double* x,
                         double* f_best, int32_t* n_eval, OrcSolveTrace* tr, double* mg) {
  const int opt_time = (mask & ORC_MINTIME) != 0;
  const int nv = opt_time ? 3 * n + 1 : 3 * n;
  const int m = sp->lbfgs_m;
  const int exact = (sp->flags & ORC_SOLVE_EXACT_EVALS) != 0;
  double X[ORC_MAXVAR], G[ORC_MAXVAR], lb[ORC_MAXVAR], ub[ORC_MAXVAR], PG[ORC_MAXVAR], D[ORC_MAXVAR],
      Q[ORC_MAXVAR], XN[ORC_MAXVAR], GN[ORC_MAXVAR], dx[ORC_MAXVAR];
  static _Thread_local double S[ORC_MAXM][ORC_MAXVAR], Y[ORC_MAXM][ORC_MAXVAR];
  double rho[ORC_MAXM] = { 0 }, alpha[ORC_MAXM];
  int act[ORC_MAXVAR];
  /* trace: mcur = smallest decision margin so far; it is written to mg[k-1] when the count leaves k */
  double mcur = INFINITY;
  OrcSolveTrace tdummy;
  if (!tr) tr = &tdummy;
  memset(tr, 0, sizeof(*tr));
  tr->first_full_reject = tr->first_ls_fail = -1;
#define NOTE(v) do { const double v_ = (v); if (!(v_ >= mcur)) mcur = v_ == v_ ? v_ : 0.0; } while (0)
#define BUMP() do { if (mg) mg[neval - 1] = mcur; ++neval; } while (0)
  for (int i = 0; i < 3 * n; ++i) {
    const int k = i % 3;
    const double bmin = g->box_mind[k] + 0.1, bmax = g->box_maxd[k] - 0.1;
    double c = x[i];
    c = fmax(fmin(c, bmax), bmin);
    X[i] = c;
    lb[i] = fmax(c - 10.0, bmin);
    ub[i] = fmin(c + 10.0, bmax);
  }
  if (opt_time) {
    X[nv - 1] = x[nv - 1];
    lb[nv - 1] = 0.0;
    ub[nv - 1] = 5.0;
  }
  double F, FN = 0.0;
  orc_combine_cost(g, dist_buf, p, tc, n, mask, X, &F, G);
  int neval = 1;
  double best = F;
  memcpy(x, X, sizeof(double) * nv);
  *f_best = F;
  if (!(best == best)) best = DBL_MAX;
  int cnt = 0, head = 0;
  while (neval < sp->max_eval) {
    for (int i = 0; i < nv; ++i) {
      act[i] = (X[i] <= lb[i] && G[i] > 0.0) || (X[i] >= ub[i] && G[i] < 0.0);
      PG[i] = act[i] ? 0.0 : G[i];
    }
    const double pgn2 = vdot(PG, PG, nv);
    NOTE(rel_margin(pgn2, 1e-24, fmax(pgn2, 1e-24)));
    if (!(pgn2 > 1e-24)) {
      if (!exact) break;
      while (neval < sp->max_eval) { /* nothing left to descend: evaluate in place */
        orc_combine_cost(g, dist_buf, p, tc, n, mask, X, &F, G);
        BUMP();
      }
      break;
    }
    memcpy(Q, PG, sizeof(double) * nv);
    for (int j = 0; j < cnt; ++j) {
      const int slot = (head - 1 - j + 2 * ORC_MAXM * m) % m;
      alpha[j] = rho[slot] * vdot(S[slot], Q, nv);
      for (int i = 0; i < nv; ++i) Q[i] -= alpha[j] * Y[slot][i];
    }
    if (cnt > 0) {
      const int slot = (head - 1 + m) % m;
      const double gamma = vdot(S[slot], Y[slot], nv) / vdot(Y[slot], Y[slot], nv);
      for (int i = 0; i < nv; ++i) Q[i] *= gamma;
    }
    for (int j = cnt - 1; j >= 0; --j) {
      const int slot = (head - 1 - j + 2 * ORC_MAXM * m) % m;
      const double beta = rho[slot] * vdot(Y[slot], Q, nv);
      for (int i = 0; i < nv; ++i) Q[i] += S[slot][i] * (alpha[j] - beta);
    }
    for (int i = 0; i < nv; ++i) D[i] = act[i] ? 0.0 : -Q[i];
    double gd = vdot(G, D, nv);
    NOTE(rel_margin(gd, 0.0, sqrt(vdot(G, G, nv) * vdot(D, D, nv))));
    if (!(gd < 0.0)) {
      for (int i = 0; i < nv; ++i) D[i] = -PG[i];
      gd = -pgn2;
      cnt = 0;
      ++tr->n_restart;
    }
    double step = cnt == 0 ? fmin(1.0, 1.0 / sqrt(pgn2)) : 1.0;
    int accepted = 0;
    while (neval < sp->max_eval) {
      for (int i = 0; i < nv; ++i) XN[i] = fmax(fmin(X[i] + step * D[i], ub[i]), lb[i]);
      orc_combine_cost(g, dist_buf, p, tc, n, mask, XN, &FN, GN);
      BUMP();
      NOTE(rel_margin(FN, best, fmax(fabs(FN), fabs(best))));
      if (FN < best) {
        best = FN;
        memcpy(x, XN, sizeof(double) * nv);
        *f_best = FN;
      }
      for (int i = 0; i < nv; ++i) dx[i] = XN[i] - X[i];
      const double dec = vdot(G, dx, nv);
      NOTE(rel_margin(FN, F + 1e-4 * dec, fmax(fabs(FN), fabs(F))));
      if (FN <= F + 1e-4 * dec) {
        accepted = 1;
        break;
      }
      step *= 0.5;
      if (step < 1e-12) break;
    }
    if (!accepted) {
      if (neval < sp->max_eval) { /* (a search cut short by the budget is not a failure) */
        ++tr->n_ls_fail;
        if (tr->first_ls_fail < 0) tr->first_ls_fail = neval;
      }
      if (!exact) break;
      cnt = 0;
      continue;
    }
    int small = 1;
    double xmargin = INFINITY, xfail = 0.0; /* xtol: the tightest component if all pass, the clearest failure if not */
    double s_[ORC_MAXVAR], y_[ORC_MAXVAR];
    for (int i = 0; i < nv; ++i) {
      s_[i] = XN[i] - X[i];
      y_[i] = GN[i] - G[i];
      const double lim = sp->xtol_rel * fabs(XN[i]);
      const int ok = fabs(s_[i]) <= lim;
      small = small && ok;
      const double mi = rel_margin(fabs(s_[i]), lim, fmax(fabs(s_[i]), lim));
      if (ok) xmargin = fmin(xmargin, mi);
      else xfail = fmax(xfail, mi);
    }
    if (!exact) NOTE(small ? xmargin : xfail);
    const double sy = vdot(s_, y_, nv), ss = vdot(s_, s_, nv), yy = vdot(y_, y_, nv);
    NOTE(rel_margin(sy, 1e-10 * sqrt(ss * yy), sqrt(ss * yy)));
    if (sy > 1e-10 * sqrt(ss * yy)) {
      memcpy(S[head], s_, sizeof(double) * nv);
      memcpy(Y[head], y_, sizeof(double) * nv);
      rho[head] = 1.0 / sy;
      head = (head + 1) % m;
      if (cnt < m) ++cnt;
      ++tr->n_kept;
    } else {
      ++tr->n_curv_reject;
      if (cnt == m) {
        ++tr->n_full_reject;
        if (tr->first_full_reject < 0) tr->first_full_reject = neval;
      }
    }
    memcpy(X, XN, sizeof(double) * nv);
    memcpy(G, GN, sizeof(double) * nv);
    F = FN;
    if (!exact && small) break;
  }
  *n_eval = neval;
  if (mg)
    for (int k = neval; k <= sp->max_eval; ++k) mg[k - 1] = mcur;
#undef NOTE
#undef BUMP
}

void orc_optimize_batch_traced(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                               const OrcTrajConst* tc, int32_t n_pts, int32_t cost_mask, int32_t B,
                               const OrcSolveParams* sp, double* x, double* f_best, int32_t* n_eval,
                               OrcSolveTrace* trace, double* margin, int threads) {
  const int nv = (cost_mask & ORC_MINTIME) ? 3 * n_pts + 1 : 3 * n_pts;
  if (threads < 1) threads = 1;
#pragma omp parallel for num_threads(threads) schedule(dynamic, 8)
  for (int b = 0; b < B; ++b)
    optimize_one(g, dist_buf, p, &tc[b], n_pts, cost_mask, sp, x + (int64_t)b * nv, &f_best[b], &n_eval[b],
                 trace ? &trace[b] : NULL, margin ? margin + (int64_t)b * sp->max_eval : NULL);
}

void orc_optimize_batch(const OrcGrid* g, const double* dist_buf, const OrcOptParams* p,
                        const OrcTrajConst* tc, int32_t n_pts, int32_t cost_mask, int32_t B,
                        const OrcSolveParams* sp, double* x, double* f_best, int32_t* n_eval,
                        int threads) {
  const int nv = (cost_mask & ORC_MINTIME) ? 3 * n_pts + 1 : 3 * n_pts;
  if (threads < 1) threads = 1;
#pragma omp parallel for num_threads(threads) schedule(dynamic, 8)
  for (int b = 0; b < B; ++b)
    optimize_one(g, dist_buf, p, &tc[b], n_pts, cost_mask, sp, x + (int64_t)b * nv, &f_best[b], &n_eval[b], NULL,
                 NULL);
}
