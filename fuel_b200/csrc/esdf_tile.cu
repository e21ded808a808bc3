// esdf_tile.cu -- the exact Euclidean distance transform as smem-resident line tiles (sm_100a).
//
// Replaces SDFMap::updateESDF3d / fillESDF (plan_env/src/sdf_map.cpp:116-241).  The reference
// runs three 1-D lower-envelope sweeps (z, y, x) in fp64 with DBL_MAX as "no site"; every finite
// intermediate is an integer (squared voxel distance <= 3*(n-1)^2), so the device keeps the
// transform in exact int32 arithmetic and only the last sweep converts: dist = res*sqrt(d2).
//
// Pipeline (box-relative coordinates, z fastest like the reference, sdf_map.h:145-147):
//   K0 zpack     occupancy bytes -> one record per 32 voxels of a z line: site bitmask + distance
//                to the nearest site below / above the word (8 B per 32 voxels, L2-resident).
//   K1 zy tile   CTA = (x, 32 consecutive z) over all y.  The records arrive by one bulk-async copy
//                (cp.async.bulk + mbarrier), are decoded to the squared z distance (exact, from the
//                bitmask) into a [y][32] shared-memory tile, and the y lower envelope runs out of
//                shared memory.  Output: the 2-D partial P (int32) of one z chunk.
//   K2 x tile    CTA = (y, 32 consecutive z) over all x.  The [x][32] tile of P is gathered by
//                bulk-async row copies, the x lower envelope runs in shared memory, result in metres.
// K1 -> K2 run per z chunk (32*Wc planes) alternating between two streams, so that P of a chunk is
// consumed out of L2 while the next chunk is produced: HBM sees 1 B in + 4 B out per voxel.
//
// Lower envelope (Felzenszwalb-Huttenlocher restated in exact integers: parabola of site v has
// height h(v) = f(v) + v^2; w overtakes u at (h(w)-h(u)) / (2(w-u)); every comparison is
// cross-multiplied, no division).  A tile holds 32 lines (lane <-> line, bank <-> lane: no
// conflicts); the line is cut into bands of 32 samples, warp <-> band, so a thread builds the hull
// of 32 samples in place (hull slot k of a band aliases the band's k-th input sample, which is dead
// by then), adjacent band hulls are joined pairwise (log2 rounds of bridge finding: with equal
// curvature the difference of the two envelopes is monotone, so the joint hull is a prefix of the
// left one followed by a suffix of the right one), and every thread evaluates its own 32 samples by
// walking the joint hull.
#include "common.cuh"

#include <stdlib.h>

namespace {

constexpr int INF_I = FUELGPU_EDT_INF_I;
constexpr int SENT = 1 << 23;   // height offset of the virtual bottom-of-stack parabola (> any real h < 2^22)
constexpr int BIGD = 0x3fff;    // "no site on this side" in the z records
constexpr int FIN_LIM = 1 << 22;  // finite squared distances are < 2^22 (2*1023^2), INF_I and BIGD^2 are above
constexpr unsigned FULL = 0xffffffffu;

struct TBox {
  int lo[3], hi[3];  // inclusive
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// shared-memory accesses by 32-bit shared-window address (the hot loops keep their cursors in this form: one
// IADD per step instead of 64-bit generic pointer arithmetic)
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  unsigned ok = 0;
  const uint32_t a = smem_u32(bar);
  while (!ok) {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
  }
}

// ---- thread-block cluster primitives (lines longer than 512 samples: one tile = 2 CTAs, hulls joined over DSMEM) ----
__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;\nbarrier.cluster.wait.acquire;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa_u32(uint32_t a, unsigned rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  return r;
}
__device__ __forceinline__ uint32_t ldc32(uint32_t ca) {
  uint32_t v;
  asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(ca) : "memory");
  return v;
}
__device__ __forceinline__ int ldc16(uint32_t ca) {
  uint16_t v;
  asm volatile("ld.shared::cluster.u16 %0, [%1];" : "=h"(v) : "r"(ca) : "memory");
  return (int)v;
}
__device__ __forceinline__ void stc16(uint32_t ca, int v) {
  asm volatile("st.shared::cluster.u16 [%0], %1;" ::"r"(ca), "h"((uint16_t)v) : "memory");
}

// site predicate of the z sweep.  mode 0: optimistic (sdf_map.cpp:156-166) inflate==1;
// mode 1: non-optimistic (:167-181) inflate==1 || unknown; mode 2: negative field (:203-214)
// inflate==0.
__device__ __forceinline__ bool is_site(uint8_t o, int mode) {
  const bool infl = (o & 4) != 0;
  if (mode == 0) return infl;
  if (mode == 1) return infl || ((o & 3) == FUELGPU_UNKNOWN);
  return !infl;
}
// the same predicate on 4 voxels at once: bit 8i of the result <-> voxel i, gathered to 4 bits
__device__ __forceinline__ uint32_t site_bits4(uint32_t w, int mode) {
  uint32_t t;
  if (mode == 0)
    t = w >> 2;
  else if (mode == 1)
    t = (w >> 2) | ~(w | (w >> 1));
  else
    t = ~(w >> 2);
  t &= 0x01010101u;
  return (t * 0x01020408u) >> 24;
}

// ---------------------------------------------------------------------------------------
// K0: rec[(x*NW + w)*NYP + y] = { site mask of word w of line (x,y), dL | dR << 16 }: dL = distance
// from bit 0 of the word to the nearest site below it (>= 1), dR = distance from bit 31 to the nearest
// site above it, BIGD if none.  One lane per 32-voxel word; a line takes LPR = 2^k >= NW lanes, so a warp
// packs 32/LPR lines.  VEC: the word is two 16-byte loads (box z range a multiple of 32 voxels on a
// 16-byte boundary); otherwise bytes are gathered with ballots, one line per warp.
// ---------------------------------------------------------------------------------------
// The z axis of a line may be split into chunks (z-sharded volume gathered from several ranks): word c lives
// in chunk c / cw at occ + (c / cw) * chunk_stride, and a chunk holds nz voxels per line (cw = words per chunk;
// one chunk with cw >= NW is the ordinary contiguous volume).
template <int MODE, bool VEC>
__global__ void __launch_bounds__(256) zpack_kernel(const uint8_t* __restrict__ occ, uint2* __restrict__ rec, int ny,
                                                    int nz, TBox b, int NW, int NYP, int lpr_log2, int cw,
                                                    int64_t chunk_stride) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nxb = b.hi[0] - b.lo[0] + 1, nyb = b.hi[1] - b.lo[1] + 1, nzb = b.hi[2] - b.lo[2] + 1;
  const int nrows = nxb * nyb;
  const int LPR = VEC ? (1 << lpr_log2) : 32;
  const int grp = VEC ? (lane >> lpr_log2) : 0;
  const int c = lane & (LPR - 1);  // word of the line this lane keeps
  const int row = VEC ? (warp << (5 - lpr_log2)) + grp : warp;
  if (!VEC && row >= nrows) return;
  const bool rvalid = row < nrows;
  const int rr = rvalid ? row : 0;
  const int xr = rr / nyb, yr = rr - xr * nyb;
  const int64_t base = ((int64_t)(b.lo[0] + xr) * ny + (b.lo[1] + yr)) * nz + b.lo[2];
  uint32_t word = 0;
  if (VEC) {
    if (rvalid && c < NW) {
      const int g = c / cw;
      const uint4* src = reinterpret_cast<const uint4*>(occ + g * chunk_stride + base + ((c - g * cw) << 5));
      const uint4 v0 = __ldg(src), v1 = __ldg(src + 1);
      word = site_bits4(v0.x, MODE) | (site_bits4(v0.y, MODE) << 4) | (site_bits4(v0.z, MODE) << 8) |
             (site_bits4(v0.w, MODE) << 12) | (site_bits4(v1.x, MODE) << 16) | (site_bits4(v1.y, MODE) << 20) |
             (site_bits4(v1.z, MODE) << 24) | (site_bits4(v1.w, MODE) << 28);
    }
  } else {
    for (int k = 0; k < NW; ++k) {
      const int p = (k << 5) + lane;
      const int g = k / cw;
      const bool s = p < nzb && is_site(__ldg(occ + g * chunk_stride + base + p - ((int64_t)g * cw << 5)), MODE);
      const uint32_t mm = __ballot_sync(FULL, s);
      if (lane == k) word = mm;
    }
  }
  const bool valid = rvalid && c < NW;
  const uint32_t ball = __ballot_sync(FULL, valid && word != 0);
  const uint32_t gb = LPR == 32 ? ball : ((ball >> (grp * LPR)) & ((1u << LPR) - 1u));
  const int mylast = word ? 31 - __clz(word) : 0;
  const int myfirst = word ? __ffs(word) - 1 : 0;
  const uint32_t pm = gb & ((1u << c) - 1u);
  const int pl = pm ? 31 - __clz(pm) : 0;
  const int plast = __shfl_sync(FULL, mylast, grp * LPR + pl);
  const uint32_t nm = gb & ~((2u << c) - 1u);
  const int nl = nm ? __ffs(nm) - 1 : 0;
  const int nfirst = __shfl_sync(FULL, myfirst, grp * LPR + nl);
  const int dL = pm ? (c << 5) - ((pl << 5) + plast) : BIGD;
  const int dR = nm ? ((nl << 5) + nfirst) - ((c << 5) + 31) : BIGD;
  if (valid) rec[((int64_t)xr * NW + c) * NYP + yr] = make_uint2(word, (uint32_t)dL | ((uint32_t)dR << 16));
}

template <int MODE>
void launch_zpack(cudaStream_t st, const uint8_t* occ, uint2* rec, int ny, int nz, const TBox& b, int NW, int NYP,
                  int cw = 1 << 20, int64_t chunk_stride = 0) {
  const int nxb = b.hi[0] - b.lo[0] + 1, nyb = b.hi[1] - b.lo[1] + 1, nzb = b.hi[2] - b.lo[2] + 1;
  const int64_t base0 = ((int64_t)b.lo[0] * ny + b.lo[1]) * nz + b.lo[2];
  const bool vec = (nzb % 32 == 0) && (nz % 16 == 0) && (base0 % 16 == 0) && (chunk_stride % 16 == 0);
  const int rows = nxb * nyb;
  if (vec) {
    int l2 = 0;
    while ((1 << l2) < NW) ++l2;
    const int rpw = 32 >> l2;  // lines per warp
    const int warps = (rows + rpw - 1) / rpw;
    zpack_kernel<MODE, true><<<(warps + 7) / 8, 256, 0, st>>>(occ, rec, ny, nz, b, NW, NYP, l2, cw, chunk_stride);
  } else {
    zpack_kernel<MODE, false><<<(rows + 7) / 8, 256, 0, st>>>(occ, rec, ny, nz, b, NW, NYP, 5, cw, chunk_stride);
  }
}

// ---------------------------------------------------------------------------------------
// K1 / K2: the line-tile envelope kernel.
// ---------------------------------------------------------------------------------------
struct TileParams {
  int n;   // samples per line
  int nb;  // bands of 32 samples = warps per CTA
  // input
  const uint2* rec;      // FROMBITS: records of (o, w0 + blockIdx.x) start at rec + (o*NW + w0 + bx)*NYP
  int NW, NYP, w0;
  // !FROMBITS: row q of the tile of (o, bx) at pin + o*in_o + bx*in_bx + (q / piece_rows)*piece_stride +
  // (q % piece_rows)*32 (int32 units): rows are contiguous inside a piece (piece_rows is a multiple of the band
  // length, or >= n for one piece)
  const int32_t* pin;
  int64_t in_o, in_bx, piece_stride;
  int piece_rows;
  // output: sample q of lane l at out + out_base + o*out_o + bx*out_bx + q*out_q + l  (int32 or float)
  void* out;
  int64_t out_base, out_o, out_bx, out_q;
  // optional: the tiles of words [k*out_tab_wl, (k+1)*out_tab_wl) go to out_tab[k] instead of `out` (bx counted from the
  // start of that group): one launch whose output is scattered over several buffers (the peers of a sharded update)
  void* out_tab[16];
  int out_tab_wl;  // 0 = unused
  int lanes_total;  // valid z positions counted from bx = 0 (lanes beyond are not stored when FINAL)
  int discard_input;  // !FROMBITS: drop the tile's lines from L2 once they are in shared memory
  float res;
};

__device__ __forceinline__ uint32_t pack_vh(int v, int h) { return ((uint32_t)v << 22) + (uint32_t)h; }
__device__ __forceinline__ int unpack_v(uint32_t e) { return (int)(e >> 22); }
__device__ __forceinline__ int unpack_h(uint32_t e) { return (int)(e & 0x3fffffu); }
__device__ __forceinline__ float fast_sqrt(float x) {
  float r;
  // a few units of 2^-24: rint((dist/res)^2) still gives back the exact integer d2 up to 2^20 (tests/helpers.py)
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Hull bookkeeping of a tile as seen by ONE lane.  LO/HI = first / one-past-last live entry of a band (row numbers of
// the whole line), ent = the entry stored in a row.  Local: this CTA's shared memory.  Remote / Cluster: the arrays of
// the other CTA of a 2-CTA cluster (rows >= rpc and bands >= nbh live in CTA 1), reached through shared::cluster.
struct HullLocal {
  uint16_t* LOl;
  uint16_t* HIl;
  uint32_t* Tl;
  int row0;  // first row held by this CTA
  __device__ __forceinline__ int lo(int b) const { return LOl[b * 32]; }
  __device__ __forceinline__ int hi(int b) const { return HIl[b * 32]; }
  __device__ __forceinline__ void set_lo(int b, int v) const { LOl[b * 32] = (uint16_t)v; }
  __device__ __forceinline__ void set_hi(int b, int v) const { HIl[b * 32] = (uint16_t)v; }
  __device__ __forceinline__ uint32_t ent(int row) const { return Tl[(row - row0) * 32]; }
  // phase 3 (row0 == 0 there)
  __device__ __forceinline__ uint32_t ent_addr(int row) const { return smem_u32(Tl) + (uint32_t)row * 128u; }
  __device__ __forceinline__ uint32_t ld(uint32_t a) const { return lds32(a); }
};
struct HullRemote {  // bands / rows of the cluster's OTHER CTA, indexed like its own HullLocal
  uint32_t LOa, HIa, Ta;  // shared::cluster addresses, lane offset included
  int row0;
  __device__ __forceinline__ int lo(int b) const { return ldc16(LOa + (uint32_t)b * 64u); }
  __device__ __forceinline__ int hi(int b) const { return ldc16(HIa + (uint32_t)b * 64u); }
  __device__ __forceinline__ void set_lo(int b, int v) const { stc16(LOa + (uint32_t)b * 64u, v); }
  __device__ __forceinline__ void set_hi(int b, int v) const { stc16(HIa + (uint32_t)b * 64u, v); }
  __device__ __forceinline__ uint32_t ent(int row) const { return ldc32(Ta + (uint32_t)(row - row0) * 128u); }
};
struct HullCluster {  // bands / rows of the whole line, whichever CTA holds them
  uint32_t LOa, HIa, Ta;  // shared::cta addresses of THIS CTA's arrays, lane offset included
  int nbh, rpc;           // bands / rows per CTA
  __device__ __forceinline__ int lo(int g) const {
    const unsigned rk = g >= nbh;
    return ldc16(mapa_u32(LOa + (uint32_t)(g - (int)rk * nbh) * 64u, rk));
  }
  __device__ __forceinline__ int hi(int g) const {
    const unsigned rk = g >= nbh;
    return ldc16(mapa_u32(HIa + (uint32_t)(g - (int)rk * nbh) * 64u, rk));
  }
  __device__ __forceinline__ uint32_t ent_addr(int row) const {
    const unsigned rk = row >= rpc;
    return mapa_u32(Ta + (uint32_t)(row - (int)rk * rpc) * 128u, rk);
  }
  __device__ __forceinline__ uint32_t ld(uint32_t a) const { return ldc32(a); }
};

// join the hull of bands [gl0, gl1) of A (left) with the hull of bands [gr0, gr1) of B (right): with equal curvature
// the difference of the two envelopes is monotone, so the joint hull is a prefix of the left one followed by a suffix
// of the right one; the bridge is found by a two-pointer walk from the junction.
template <class HA, class HB>
__device__ __forceinline__ void join_hulls(const HA& A, int gl0, int gl1, const HB& B, int gr0, int gr1) {
  int bl = gl1 - 1;
  while (bl >= gl0 && A.lo(bl) == A.hi(bl)) --bl;
  int br = gr0;
  while (br < gr1 && B.lo(br) == B.hi(br)) ++br;
  if (bl < gl0 || br >= gr1) return;
  int il = A.hi(bl) - 1, jr = B.lo(br);
  uint32_t e = A.ent(il);
  int vi = unpack_v(e), hi_ = unpack_h(e);
  e = B.ent(jr);
  int vj = unpack_v(e), hj = unpack_h(e);
  // predecessor of the left end / successor of the right end inside their groups
  int pb = bl, pi = il - 1, vp = 0, hp = 0;
  bool hasp;
  int nbd = br, ni = jr + 1, vn = 0, hn = 0;
  bool hasn;
  auto find_prev = [&]() {
    if (pi < A.lo(pb)) {
      --pb;
      while (pb >= gl0 && A.lo(pb) == A.hi(pb)) --pb;
      if (pb >= gl0) pi = A.hi(pb) - 1;
    }
    hasp = pb >= gl0;
    if (hasp) {
      const uint32_t ee = A.ent(pi);
      vp = unpack_v(ee);
      hp = unpack_h(ee);
    }
  };
  auto find_next = [&]() {
    if (ni >= B.hi(nbd)) {
      ++nbd;
      while (nbd < gr1 && B.lo(nbd) == B.hi(nbd)) ++nbd;
      if (nbd < gr1) ni = B.lo(nbd);
    }
    hasn = nbd < gr1;
    if (hasn) {
      const uint32_t ee = B.ent(ni);
      vn = unpack_v(ee);
      hn = unpack_h(ee);
    }
  };
  find_prev();
  find_next();
  while (true) {
    const long long A_ = (long long)(hj - hi_);
    const long long dji = (long long)(vj - vi);
    if (hasp && A_ * (long long)(vi - vp) <= (long long)(hi_ - hp) * dji) {
      // the left end never gets below the right hull inside its own region: drop it
      il = pi;
      bl = pb;
      vi = vp;
      hi_ = hp;
      pi = il - 1;
      find_prev();
      continue;
    }
    if (hasn && A_ * (long long)(vn - vj) >= (long long)(hn - hj) * dji) {
      jr = ni;
      br = nbd;
      vj = vn;
      hj = hn;
      ni = jr + 1;
      find_next();
      continue;
    }
    break;
  }
  for (int b2 = bl + 1; b2 < gl1; ++b2) A.set_hi(b2, A.lo(b2));
  A.set_hi(bl, il + 1);
  for (int b2 = gr0; b2 < br; ++b2) B.set_lo(b2, B.hi(b2));
  B.set_lo(br, jr);
}

// phase 3: the thread of band `gband` (samples [j0, qend)) evaluates its samples on the joint hull of all nbt bands
template <bool FINAL, int LOGM, class H>
__device__ __forceinline__ void evaluate_band(const H& hull, int gband, int nbt, int j0, int qend, char* op,
                                              unsigned ostride, float res) {
  int cb = gband;
  while (cb >= 0 && hull.lo(cb) == hull.hi(cb)) --cb;
  bool empty = false;
  if (cb < 0) {
    cb = gband + 1;
    while (cb < nbt && hull.lo(cb) == hull.hi(cb)) ++cb;
    empty = cb >= nbt;
  } else {
    // go back while the first entry of band cb has not yet taken over from its predecessor at j0
    while (true) {
      int pb = cb - 1;
      while (pb >= 0 && hull.lo(pb) == hull.hi(pb)) --pb;
      if (pb < 0) break;
      const uint32_t e1 = hull.ld(hull.ent_addr(hull.lo(cb))), e0 = hull.ld(hull.ent_addr(hull.hi(pb) - 1));
      if (unpack_h(e1) - unpack_h(e0) < 2 * j0 * (unpack_v(e1) - unpack_v(e0))) break;
      cb = pb;
    }
  }
  if (empty) {
    for (int u = 0; u < qend - j0; ++u) {
      char* const a = op + (uint64_t)(unsigned)u * ostride;
      if (FINAL)
        *reinterpret_cast<float*>(a) = __int_as_float(0x7f800000);
      else
        *reinterpret_cast<int32_t*>(a) = INF_I;
    }
    return;
  }
  // cur = (vc,hc); np -> the entry after it, nend = end of np's band; (dvn,dhn) = next - cur, or (0,1) when
  // the hull is exhausted (the takeover test 2q*dvn > dhn can then never fire)
  uint32_t np, nend;
  {
    const int l0 = hull.lo(cb);
    np = hull.ent_addr(l0);
    nend = np + (uint32_t)(hull.hi(cb) - l0) * 128u;
  }
  int vc, hc, dvn, dhn;
  {
    const uint32_t e = hull.ld(np);
    vc = unpack_v(e);
    hc = unpack_h(e);
  }
  // advance np to the following live entry; false when there is none
  auto step_next = [&]() -> bool {
    np += 128u;
    if (np == nend) {
      ++cb;
      while (cb < nbt && hull.lo(cb) == hull.hi(cb)) ++cb;
      if (cb >= nbt) return false;
      const int l0 = hull.lo(cb);
      np = hull.ent_addr(l0);
      nend = np + (uint32_t)(hull.hi(cb) - l0) * 128u;
    }
    return true;
  };
  if (step_next()) {
    const uint32_t e = hull.ld(np);
    dvn = unpack_v(e) - vc;
    dhn = unpack_h(e) - hc;
  } else {
    dvn = 0;
    dhn = 1;
  }
  const int cnt = qend - j0;
  // val(q) = (q-vc)^2 + f(vc) = hc + q(q - 2vc) is carried incrementally: val(q+1) = val(q) + inc, inc += 2
  int val = hc + j0 * (j0 - 2 * vc), inc = 2 * (j0 - vc) + 1;
  char* oa = op;
#pragma unroll 2
  for (int u = 0; u < cnt; ++u) {
    const int q = j0 + u;
    // the next parabola takes over at the first integer q with (hn-hc) < 2q(vn-vc)
    if (2 * q * dvn > dhn) {
      do {
        vc += dvn;
        hc += dhn;
        if (!step_next()) {
          dvn = 0;
          dhn = 1;
          break;
        }
        const uint32_t e = hull.ld(np);
        dvn = unpack_v(e) - vc;
        dhn = unpack_h(e) - hc;
      } while (2 * q * dvn > dhn);
      val = hc + q * (q - 2 * vc);
      inc = 2 * (q - vc) + 1;
    }
    if (FINAL)
      *reinterpret_cast<float*>(oa) = res * fast_sqrt((float)val);
    else
      *reinterpret_cast<int32_t*>(oa) = val;
    oa += ostride;
    val += inc;
    inc += 2;
  }
}

// CL: the tile of a line longer than 512 samples is shared by the two CTAs of a thread-block cluster (CTA r holds
// rows [r*rpc, (r+1)*rpc): 64 KB each, three CTAs per SM instead of one 128 KB CTA); p.nb = bands per CTA.
template <bool FROMBITS, bool FINAL, int LOGM, int MAXT, int MINB, bool CL>
__global__ void __launch_bounds__(MAXT, MINB) envelope_tile_kernel(const TileParams p) {
  constexpr int M = 1 << LOGM;  // samples per band (= per thread)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int n = p.n, nb = p.nb;
  uint32_t* const T = reinterpret_cast<uint32_t*>(smem_raw);                 // [nb*M][32]
  uint16_t* const LO = reinterpret_cast<uint16_t*>(T + (size_t)nb * M * 32);  // [nb][32]
  uint16_t* const HI = LO + nb * 32;                                         // [nb][32]
  uint64_t* const bar = reinterpret_cast<uint64_t*>(HI + nb * 32);
  uint2* const side = reinterpret_cast<uint2*>(bar + 2);                     // FROMBITS: [nb*M]

  const int lane = threadIdx.x & 31;
  const int band = threadIdx.x >> 5;
  const unsigned rank = CL ? cluster_ctarank() : 0u;
  const int bx = CL ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, o = blockIdx.y;
  const int rpc = nb << LOGM;                 // rows per CTA
  const int row0 = CL ? (int)rank * rpc : 0;  // first row of the line held here
  const int gband = (CL ? (int)rank * nb : 0) + band;
  uint32_t* const Tl = T + lane;
  uint16_t* const LOl = LO + lane;
  uint16_t* const HIl = HI + lane;
  const int j0 = gband << LOGM;  // first sample (row of the line) of this thread's band
  const int nloc = max(0, min(n - row0, rpc));  // rows of the line held here

  // ---- phase 0: bring the tile in ----------------------------------------------------
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  if (FROMBITS) {
    if (threadIdx.x == 0) {
      const unsigned bytes = (unsigned)(((nloc * 8) + 15) & ~15);
      mbar_expect_tx(bar, bytes);
      if (bytes) bulk_g2s(side, p.rec + ((int64_t)o * p.NW + p.w0 + bx) * p.NYP + row0, bytes, bar);
    }
    // one warp polls the mbarrier, the others sleep at the CTA barrier (a spinning try_wait in every
    // warp took 46 % of the issue slots of the SM away from the CTAs that had work)
    if (band == 0) mbar_wait(bar, 0);
    __syncthreads();
    // decode: thread t <-> sample (row) t of its own band.  The 32 squared z distances of a row are
    // produced by two running scans over the mask and written column-rotated (value i of row t at
    // column i ^ (t & 31)) so that the 32 rows of a warp hit 32 different banks; phase 1 reads its
    // input through the same rotation.  "No site" comes out as a square >= 2^26 (> FIN_LIM).
#pragma unroll 1
    for (int rep = 0; rep < M / 32; ++rep) {
      const int t = j0 + rep * 32 + lane;  // rows of this warp's own band; rotation = t & 31 = lane
      uint32_t m = 0;
      int dl = BIGD, dr = BIGD;
      if (t < n) {
        const uint2 r = side[t - row0];
        m = r.x;
        dl = (int)(r.y & 0xffffu);
        dr = (int)(r.y >> 16);
      }
      uint32_t* const Trow = T + (size_t)(t - row0) * 32;
      if (__all_sync(FULL, m == 0)) {
        // no site inside this word for any of the warp's 32 rows (the common case in open space)
        if (__all_sync(FULL, dl >= BIGD && dr >= BIGD)) {
#pragma unroll
          for (int i = 0; i < 32; ++i) Trow[i ^ lane] = (uint32_t)INF_I;
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int d = min(dl + i, dr + 31 - i);
            Trow[i ^ lane] = (uint32_t)(d * d);
          }
        }
        continue;
      }
      int dleft[32];
      dl -= 1;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        dl = ((m >> i) & 1u) ? 0 : dl + 1;
        dleft[i] = dl;
      }
      dr -= 1;
#pragma unroll
      for (int i = 31; i >= 0; --i) {
        dr = ((m >> i) & 1u) ? 0 : dr + 1;
        const int d = min(dleft[i], dr);
        Trow[i ^ lane] = (uint32_t)(d * d);
      }
    }
    __syncwarp();
  } else {
    // the tile is contiguous in P (K1 writes it that way): every warp brings its own band in with ONE bulk copy
    if (threadIdx.x == 0) mbar_expect_tx(bar, (unsigned)nloc * 128u);
    const int piece = j0 / p.piece_rows;
    const int32_t* const bsrc = p.pin + (int64_t)o * p.in_o + (int64_t)bx * p.in_bx + (int64_t)piece * p.piece_stride +
                                (int64_t)(j0 - piece * p.piece_rows) * 32;
    if (lane == 0 && j0 < n)
      bulk_g2s(T + (size_t)(j0 - row0) * 32, bsrc, (unsigned)(min(n, j0 + M) - j0) * 128u, bar);
    if (band == 0) mbar_wait(bar, 0);
    __syncthreads();
    // the tile of P is dead once it sits in shared memory: drop its lines from L2 instead of letting them be
    // written back to HBM later (P is produced and consumed out of L2; only the fp32 result should reach DRAM)
    if (p.discard_input)
      for (int r = lane; r < min(M, n - j0); r += 32)
        asm volatile("discard.global.L2 [%0], 128;" ::"l"(reinterpret_cast<const char*>(bsrc) + (size_t)r * 128)
                     : "memory");
  }

  // ---- phase 1: hull of the band's own 32 samples, in place --------------------------------
  {
    int v1 = j0 - 1, h1 = SENT + v1 * v1;  // virtual bottom parabola, never stored, owns nothing in [0,n)
    int dv = 1, dh = -2 * SENT;
    const uint32_t lane4 = (uint32_t)lane * 4u;
    const uint32_t slot0 = smem_u32(T) + (uint32_t)(j0 - row0) * 128u + lane4;  // byte address of this line's slot 0
    uint32_t slot = slot0;  // next free slot; entries so far = (slot - slot0) / 128
    uint32_t rowa = smem_u32(T) + (uint32_t)(j0 - row0) * 128u;  // row q of the tile
    uint32_t u4 = 0;                                     // 4 * (q & 31): rotation of row q (FROMBITS)
    const int qend = min(n, j0 + M);
    const int n2m2 = 2 * (n - 1);
    // (rolled on purpose: the fully unrolled kernel was 83 KB of SASS and ran out of the instruction cache)
#pragma unroll 2
    for (int q = j0; q < qend; ++q) {
      {
        // (the band's rows were decoded by this warp itself: value of lane l sits at column l ^ (q & 31))
        const int f = (int)lds32(FROMBITS ? (rowa | (lane4 ^ u4)) : (rowa + lane4));
        rowa += 128u;
        u4 = (u4 + 4u) & 124u;
        if (FROMBITS) __syncwarp();  // all lanes have read row q before any of them reuses it as a hull slot
        if (f < FIN_LIM) {
          const int h = f + q * q;
          int a = h - h1, b = q - v1;
          // q gets below the current top only at x > a/(2b): beyond the last sample it can never matter
          // (everything older is already above the top there), so it is not even pushed
          if (a >= b * n2m2) continue;
          // pop while  s(top,q) <= s(second,top):  (h-h1)*(v1-v0) <= (h1-h0)*(q-v1)
          while (a * dv <= dh * b) {
            slot -= 128u;
            v1 -= dv;
            h1 -= dh;
            if (slot >= slot0 + 256u) {
              const uint32_t e = lds32(slot - 256u);
              dv = v1 - unpack_v(e);
              dh = h1 - unpack_h(e);
            } else if (slot == slot0 + 128u) {  // the virtual bottom is second now
              dv = v1 - (j0 - 1);
              dh = h1 - (SENT + (j0 - 1) * (j0 - 1));
            } else {  // the virtual bottom is on top
              dv = 1;
              dh = -2 * SENT;
            }
            a = h - h1;
            b = q - v1;
          }
          sts32(slot, pack_vh(q, h));
          slot += 128u;
          dv = b;
          dh = a;
          v1 = q;
          h1 = h;
        }
      }
    }
    LOl[band * 32] = (uint16_t)j0;
    HIl[band * 32] = (uint16_t)(j0 + (int)((slot - slot0) >> 7));
  }

  // ---- phase 2: join adjacent hulls pairwise ---------------------------------------------
  const HullLocal loc = { LOl, HIl, Tl, row0 };
  for (int s = 1; s < nb; s <<= 1) {
    __syncthreads();
    if ((band & (2 * s - 1)) == 0 && band + s < nb) join_hulls(loc, band, band + s, loc, band + s, min(band + 2 * s, nb));
  }
  if (CL) {
    // the two halves of the line: CTA 0 walks its own hull from the top and CTA 1's from the bottom over DSMEM
    cluster_sync_all();
    if (rank == 0 && band == 0) {
      const HullRemote rem = { mapa_u32(smem_u32(LOl), 1u), mapa_u32(smem_u32(HIl), 1u), mapa_u32(smem_u32(Tl), 1u), rpc };
      join_hulls(loc, 0, nb, rem, 0, nb);
    }
    cluster_sync_all();
  } else {
    __syncthreads();
  }

  // ---- phase 3: every thread evaluates its own 32 samples on the joint hull -----------------
  if (j0 < n && !(FINAL && bx * 32 + lane >= p.lanes_total)) {  // (padding lane of the last z word: nothing to store)
    const int qend = min(n, j0 + M);
    char* outp = reinterpret_cast<char*>(p.out);
    int bxo = bx;
    if (!FINAL && p.out_tab_wl > 0) {
      const int k = bx / p.out_tab_wl;
      outp = reinterpret_cast<char*>(p.out_tab[k]);
      bxo = bx - k * p.out_tab_wl;
    }
    const int64_t obase = p.out_base + (int64_t)o * p.out_o + (int64_t)bxo * p.out_bx + lane + (int64_t)j0 * p.out_q;
    // sample j0+u goes to op + u*ostride bytes (the stride fits 32 bits: one IMAD.WIDE per store)
    char* const op = outp + obase * 4;
    const unsigned ostride = (unsigned)p.out_q * 4u;
    if (CL) {
      const HullCluster hull = { smem_u32(LOl), smem_u32(HIl), smem_u32(Tl), nb, rpc };
      evaluate_band<FINAL, LOGM>(hull, gband, 2 * nb, j0, qend, op, ostride, p.res);
    } else {
      evaluate_band<FINAL, LOGM>(loc, gband, nb, j0, qend, op, ostride, p.res);
    }
  }
  // a CTA's shared memory must outlive the other CTA's walks through it
  if (CL) cluster_sync_all();
}

size_t tile_smem_bytes(int nb, int m, bool frombits) {
  size_t s = (size_t)nb * m * 32 * 4 + (size_t)nb * 32 * 2 * 2 + 16;
  if (frombits) s += (size_t)nb * m * 8 + 16;
  return s;
}

int g_band_log2 = -1;  // FUELGPU_ESDF_BAND=64 selects 64-sample bands (default 32)
bool g_use_cluster = true;  // FUELGPU_ESDF_CLUSTER=0: long lines as one 1024-thread CTA per tile (the older form)

template <bool FROMBITS, bool FINAL>
cudaError_t launch_tile(cudaStream_t st, TileParams p, int gx, int gy) {
  if (g_band_log2 < 0) {
    const char* e = getenv("FUELGPU_ESDF_BAND");
    g_band_log2 = (e && atoi(e) == 64) ? 6 : 5;  // 32 measured faster (more warps per tile: 0.66 vs 0.68 ms at 512^3)
    const char* c = getenv("FUELGPU_ESDF_CLUSTER");
    g_use_cluster = !(c && atoi(c) == 0);
  }
  // bands of 64 samples halve the per-thread fixed work (hull joins, start search) but also the warps per tile
  const int logm = (p.n > 128 && g_band_log2 == 6 && (FROMBITS || p.piece_rows % 64 == 0)) ? 6 : 5;
  const int m = 1 << logm;
  const int nb = (p.n + m - 1) / m;
  // lines longer than 512 samples: the tile is split over the two CTAs of a cluster (64 KB each, 3 CTAs per SM)
  // instead of one 128 KB CTA that owns the SM alone
  const bool cl = logm == 5 && nb > 16 && g_use_cluster && (FROMBITS || p.piece_rows % 32 == 0);
  p.nb = cl ? (nb + 1) / 2 : nb;
  const size_t smem = tile_smem_bytes(p.nb, m, FROMBITS);
  dim3 grid((unsigned)(cl ? 2 * gx : gx), (unsigned)gy);
#define FUEL_TILE_LAUNCH(LOGM, MAXT, MINB, CLUSTER)                                                        \
  do {                                                                                                     \
    auto kfn = envelope_tile_kernel<FROMBITS, FINAL, LOGM, MAXT, MINB, CLUSTER>;                           \
    static bool attr_done = false;                                                                         \
    if (!attr_done) {                                                                                      \
      cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);  \
      if (e != cudaSuccess) return e;                                                                      \
      attr_done = true;                                                                                    \
    }                                                                                                      \
    if (CLUSTER) {                                                                                         \
      cudaLaunchConfig_t cfg;                                                                              \
      memset(&cfg, 0, sizeof(cfg));                                                                        \
      cfg.gridDim = grid;                                                                                  \
      cfg.blockDim = dim3((unsigned)p.nb * 32);                                                            \
      cfg.dynamicSmemBytes = smem;                                                                         \
      cfg.stream = st;                                                                                     \
      cudaLaunchAttribute at[1];                                                                           \
      at[0].id = cudaLaunchAttributeClusterDimension;                                                      \
      at[0].val.clusterDim.x = 2;                                                                          \
      at[0].val.clusterDim.y = 1;                                                                          \
      at[0].val.clusterDim.z = 1;                                                                          \
      cfg.attrs = at;                                                                                      \
      cfg.numAttrs = 1;                                                                                    \
      cudaError_t e = cudaLaunchKernelEx(&cfg, kfn, p);                                                    \
      if (e != cudaSuccess) return e;                                                                      \
    } else {                                                                                               \
      kfn<<<grid, p.nb * 32, smem, st>>>(p);                                                               \
    }                                                                                                      \
  } while (0)
  if (cl) {
    FUEL_TILE_LAUNCH(5, 512, 3, true);
  } else if (logm == 5) {
    if (nb <= 8)
      FUEL_TILE_LAUNCH(5, 256, 6, false);
    else if (nb <= 16)
      FUEL_TILE_LAUNCH(5, 512, 3, false);
    else
      FUEL_TILE_LAUNCH(5, 1024, 1, false);
  } else {
    if (nb <= 8)
      FUEL_TILE_LAUNCH(6, 256, 3, false);
    else
      FUEL_TILE_LAUNCH(6, 512, 1, false);
  }
#undef FUEL_TILE_LAUNCH
  return cudaGetLastError();
}

}  // namespace

// scratch the transform needs for a map of extent (nx,ny,nz): records + two P chunk buffers
void esdf_tile_scratch_sizes(int nx, int ny, int nz, size_t* rec_bytes, size_t* p_bytes, int* wc) {
  const int NW = (nz + 31) / 32, NYP = (ny + 1) & ~1;
  *rec_bytes = (size_t)nx * NW * NYP * 8 + 64;
  const size_t per_word = (size_t)nx * ny * 128;
  int w = NW;
  if (per_word * NW > (size_t)48 << 20) {
    w = (int)(((size_t)32 << 20) / per_word);
    if (w < 1) w = 1;
  }
  *wc = w;
  *p_bytes = per_word * w;
}

// one transform of the box: sites per `mode`, result (metres, +inf where the box has no site) into out
int esdf_tile_transform(FuelMap* m, const int lo[3], const int hi[3], int mode, float* out) {
  TBox b;
  for (int i = 0; i < 3; ++i) {
    b.lo[i] = lo[i];
    b.hi[i] = hi[i];
  }
  const int nxb = hi[0] - lo[0] + 1, nyb = hi[1] - lo[1] + 1, nzb = hi[2] - lo[2] + 1;
  const int ny = m->g.ny, nz = m->g.nz;
  const int NW = (nzb + 31) / 32, NYP = (nyb + 1) & ~1;
  uint2* rec = (uint2*)m->esdf_rec;
  cudaStream_t s0 = m->stream, s1 = m->esdf_aux;

  // K0
  {
    if (mode == 0)
      launch_zpack<0>(s0, m->occ, rec, ny, nz, b, NW, NYP);
    else if (mode == 1)
      launch_zpack<1>(s0, m->occ, rec, ny, nz, b, NW, NYP);
    else
      launch_zpack<2>(s0, m->occ, rec, ny, nz, b, NW, NYP);
    FUEL_LAUNCHES(m, 1);
  }
  // chunks of Wc words
  const size_t per_word = (size_t)nxb * nyb * 128;
  int Wc = NW;
  if (per_word * NW > (size_t)48 << 20) {
    Wc = (int)(((size_t)32 << 20) / per_word);
    if (Wc < 1) Wc = 1;
  }
  if (per_word * Wc > m->esdf_p_bytes) Wc = (int)(m->esdf_p_bytes / per_word);
  if (Wc < 1) return fuel_fail(m, FUELGPU_ENOMEM, "ESDF scratch too small for the box");
  const int nchunks = (NW + Wc - 1) / Wc;
  const bool two = nchunks > 1;
  if (two) {
    FUEL_CUDA(m, cudaEventRecord(m->esdf_ev[0], s0));
    FUEL_CUDA(m, cudaStreamWaitEvent(s1, m->esdf_ev[0], 0));
  }
  for (int c = 0; c < nchunks; ++c) {
    cudaStream_t st = (c & 1) ? s1 : s0;
    int32_t* P = (int32_t*)m->esdf_p[c & 1];
    const int w0 = c * Wc, wn = min(Wc, NW - w0);
    TileParams p1;
    memset(&p1, 0, sizeof(p1));
    p1.n = nyb;
    p1.rec = rec;
    p1.NW = NW;
    p1.NYP = NYP;
    p1.w0 = w0;
    p1.out = P;
    // P chunk layout [y][w][x][32]: the K2 tile of (y, w) is one contiguous run of nxb*128 bytes
    p1.out_base = 0;
    p1.out_o = 32;
    p1.out_bx = (int64_t)nxb * 32;
    p1.out_q = (int64_t)wn * nxb * 32;
    p1.lanes_total = 1 << 30;
    FUEL_CUDA(m, (launch_tile<true, false>(st, p1, wn, nxb)));
    TileParams p2;
    memset(&p2, 0, sizeof(p2));
    p2.n = nxb;
    p2.pin = P;
    p2.in_o = (int64_t)wn * nxb * 32;
    p2.in_bx = (int64_t)nxb * 32;
    p2.piece_rows = 1 << 20;
    p2.piece_stride = 0;
    p2.discard_input = 1;
    p2.out = out;
    p2.out_base = ((int64_t)lo[0] * ny + lo[1]) * nz + lo[2] + (int64_t)w0 * 32;
    p2.out_o = nz;
    p2.out_bx = 32;
    p2.out_q = (int64_t)ny * nz;
    p2.lanes_total = nzb - w0 * 32;
    p2.res = (float)m->g.res;
    FUEL_CUDA(m, (launch_tile<false, true>(st, p2, wn, nyb)));
    FUEL_LAUNCHES(m, 2);
  }
  if (two) {
    FUEL_CUDA(m, cudaEventRecord(m->esdf_ev[1], s1));
    FUEL_CUDA(m, cudaStreamWaitEvent(s0, m->esdf_ev[1], 0));
  }
  return 0;
}


// ---- stage launchers for the sharded update (sharded.cu): explicit layouts, caller-owned buffers -------------
// records of a [nxl][ny][G*nzc] volume whose z axis arrives as G chunks of nzc planes (chunk g at occ + g*chunk_stride)
int edt_stage_zpack(cudaStream_t st, const uint8_t* occ, void* rec, int nxl, int ny, int nzc, int G, int64_t chunk_stride,
                    int mode) {
  TBox b;
  b.lo[0] = b.lo[1] = b.lo[2] = 0;
  b.hi[0] = nxl - 1;
  b.hi[1] = ny - 1;
  b.hi[2] = G * nzc - 1;
  const int NW = (G * nzc + 31) / 32, NYP = (ny + 1) & ~1;
  if (G > 1 && nzc % 32) return FUELGPU_EINVAL;
  const int cw = G > 1 ? nzc / 32 : 1 << 20;
  if (mode == 0)
    launch_zpack<0>(st, occ, (uint2*)rec, ny, nzc, b, NW, NYP, cw, chunk_stride);
  else if (mode == 1)
    launch_zpack<1>(st, occ, (uint2*)rec, ny, nzc, b, NW, NYP, cw, chunk_stride);
  else
    launch_zpack<2>(st, occ, (uint2*)rec, ny, nzc, b, NW, NYP, cw, chunk_stride);
  return cudaGetLastError() == cudaSuccess ? 0 : FUELGPU_ECUDA;
}

// zy tiles of words [w0, w0+wn) for all nxl planes; sample (x, y, w, lane) goes to P[x*out_o + (w-w0)*out_bx + y*out_q + lane]
int edt_stage_zy(cudaStream_t st, const void* rec, int nxl, int ny, int NW, int w0, int wn, int32_t* P, int64_t out_o,
                 int64_t out_bx, int64_t out_q) {
  TileParams p1;
  memset(&p1, 0, sizeof(p1));
  p1.n = ny;
  p1.rec = (const uint2*)rec;
  p1.NW = NW;
  p1.NYP = (ny + 1) & ~1;
  p1.w0 = w0;
  p1.out = P;
  p1.out_o = out_o;
  p1.out_bx = out_bx;
  p1.out_q = out_q;
  p1.lanes_total = 1 << 30;
  return launch_tile<true, false>(st, p1, wn, nxl) == cudaSuccess ? 0 : FUELGPU_ECUDA;
}

// the same for ALL words of the line at once, scattered over ntab output buffers: words [k*wl, (k+1)*wl) go to tab[k]
// with the word index counted from k*wl (ntab <= 16)
int edt_stage_zy_scatter(cudaStream_t st, const void* rec, int nxl, int ny, int NW, int32_t* const* tab, int ntab, int wl,
                         int64_t out_o, int64_t out_bx, int64_t out_q) {
  if (ntab < 1 || ntab > 16 || ntab * wl != NW) return FUELGPU_EINVAL;
  TileParams p1;
  memset(&p1, 0, sizeof(p1));
  p1.n = ny;
  p1.rec = (const uint2*)rec;
  p1.NW = NW;
  p1.NYP = (ny + 1) & ~1;
  p1.w0 = 0;
  p1.out = tab[0];
  for (int k = 0; k < ntab; ++k) p1.out_tab[k] = tab[k];
  p1.out_tab_wl = wl;
  p1.out_o = out_o;
  p1.out_bx = out_bx;
  p1.out_q = out_q;
  p1.lanes_total = 1 << 30;
  return launch_tile<true, false>(st, p1, NW, nxl) == cudaSuccess ? 0 : FUELGPU_ECUDA;
}

// x tiles: grid (wn, ny); tile rows per TileParams (pieces); result in metres to out[y*out_o + w*out_bx + x*out_q + lane]
int edt_stage_x(cudaStream_t st, const int32_t* P, int64_t in_o, int64_t in_bx, int64_t piece_stride, int piece_rows, int nx,
                int ny, int wn, float* out, int64_t out_o, int64_t out_bx, int64_t out_q, int lanes_total, float res,
                int discard) {
  TileParams p2;
  memset(&p2, 0, sizeof(p2));
  p2.n = nx;
  p2.pin = P;
  p2.in_o = in_o;
  p2.in_bx = in_bx;
  p2.piece_stride = piece_stride;
  p2.piece_rows = piece_rows;
  p2.discard_input = discard;
  p2.out = out;
  p2.out_o = out_o;
  p2.out_bx = out_bx;
  p2.out_q = out_q;
  p2.lanes_total = lanes_total;
  p2.res = res;
  return launch_tile<false, true>(st, p2, wn, ny) == cudaSuccess ? 0 : FUELGPU_ECUDA;
}
