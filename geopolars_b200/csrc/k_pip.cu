// k_pip.cu — points-in-polygons broadcast join: the north-star path
// ("100M random points .contains() against 10k 64-vertex polygons", BASELINE.json configs[1]).
//
// Reference semantics (file:line under /root/reference):
//   * candidate generation = bbox overlap with closed intervals (rstar AABB,
//     geopolars/src/spatial_index.rs:74-76, 206-312),
//   * exact test = `poly.contains(point)` for every predicate (spatial_index.rs:89-96), i.e. geo 0.27
//     coordinate_position == Inside: winding number with exact orient2d, boundary => NOT contained
//     (pinned by the 9-point vector at spatial_index.rs:432-484),
//   * output = (lhs_index, rhs_index) pairs (spatial_index.rs:139-157).
//
// B200 design.  The polygon side is small (10 MB) and lives in the 126 MB L2; the point side is a 1.6 GB
// stream.  Round 1 walked an edge list for EVERY point (two dependent L2 gathers + ~10 edge rules per point,
// 20 of 32 lanes active, 0.15 of the HBM roofline).  Round 2 answers most points from a 2-bit raster:
//
//   fine cell (arithmetic)  -> 2-bit code from an L2-resident raster (64-bit words: the codes of 16 cells + the
//                              polygon row of the coarse cell's candidate #0):
//                                0 = outside every polygon                       -> id -1, done
//                                1 / 2 = strictly inside the coarse cell's candidate #0 / #1 and
//                                        outside every other polygon              -> id from the word (1) or an
//                                                                                    8-byte record (2), done
//                                3 = a ring passes through (or near) the cell, or anything else -> WALK
//   WALK (~13 % of the points on config 2): the point is appended to a per-warp shared-memory queue and the
//   queue is drained 32 points at a time, so that the edge walk runs with full warps:
//   coarse cell             -> ONE 32-byte record = candidate count + the first candidate's x-range and
//                              y-bucket parameters (one 256-bit load)
//   y-bucket (arithmetic)   -> plain parts: fixed-stride FP32 table, header + edges as 16-byte float records;
//                              other parts: (start,end) of a list of 32-byte f64 edge records
//   edge rule               -> branch-free; an FP32 filter with a rigorous error bound on the fast table, the
//                              f64 determinant with Shewchuk's stage-A filter elsewhere; whatever a filter
//                              cannot certify is appended to a list and recomputed exactly by a second kernel.
//
// Exactness of the pruning: geo's loop only ever acts on an edge when p.y lies in the edge's closed
// y-range.  Buckets are assigned with f(y) = clamp(floor((y - ymin) * inv_h)), a monotone
// non-decreasing function of y in IEEE arithmetic (subtraction, multiplication by a positive constant,
// floor and clamp are all monotone), and an edge is listed in buckets f(ylo)..f(yhi); hence
// ylo <= p.y <= yhi implies the edge is in bucket f(p.y): the bucket list is a superset of the edges
// the reference would act on, and every listed edge is evaluated with the reference's own rule.
// The same argument covers the grid cells (bbox filter).  No epsilon anywhere in the pruning.
//
// Exactness of the raster (see "raster" below): a cell keeps a code other than 3 only if no ring segment of ANY
// part comes within 1e-6 cell widths of it; such a cell lies inside one face of every part's ring arrangement, so
// one exact test of one representative point (geo's rule, adaptive orient2d) classifies every point that maps to
// the cell.  Points on or near a boundary always take the walk, i.e. geo's own rule.
#include <cooperative_groups.h>
#include <math.h>
#include <string.h>

#include "common.cuh"
#include "scan.cuh"

namespace cg = cooperative_groups;

namespace gpl {

struct __align__(16) PartHeader {  // build-time record (double-precision bbox), 64 bytes
    double xmin, ymin, xmax, ymax;
    double inv_h;          // (double)(float)(n_buckets / (ymax - by0)), 0 when degenerate
    int32_t n_buckets;
    int32_t bucket_base;   // first bucket of this part in bucket_start[]
    int32_t geom;          // parent row in the polygon array
    int32_t flags;         // bit0: has holes (entries carry ring ids), bit1: valid
    double by0;            // bucket origin: (double)float_round_down(ymin)
};
static_assert(sizeof(PartHeader) == 64, "PartHeader must be 64 bytes");

// Query-time part parameters (24 bytes).  All FLOAT, all CONSERVATIVE:
//   xminf/xmaxf  the x-range rounded outwards: can only fail to reject, never reject a point inside;
//   yminf        the bucket origin, ymin rounded DOWN;  inv_hf = n_buckets / (ymax - yminf).
// The bucket function f(y) = min(floor((y - yminf) * inv_hf), nb-1) is evaluated in double on these
// float-valued parameters, identically at build and query time, so it is the same monotone function
// on both sides (that is all the exactness argument needs).  t < 0 <=> y < yminf <= ymin, and
// t >= nb + 1 implies y > ymax (inv_hf carries a relative error of 2^-23, nb <= 4096).
struct PartLite {
    float xminf, xmaxf, yminf, inv_hf;
    int32_t nb_flags;     // n_buckets in bits 0..23, bit 31: part has holes
    int32_t bucket_base;
};
// one 32-byte sector per part: parameters + parent row (candidates after the first of a cell)
struct __align__(32) PartRec {
    PartLite lite;
    int32_t geom;
    int32_t pad;
};
static_assert(sizeof(PartRec) == 32, "PartRec must be one sector");

// coarse grid cell: one sector.  count == 1: `first` is the part id and `lite` its parameters — the common
// case costs a single 256-bit load.  count > 1: `first` is the offset of the ascending part-id list in
// cell_items[], `lite` belongs to the first (lowest) of them.
struct __align__(32) CellRec {
    int32_t count;
    int32_t first;
    PartLite lite;
};
static_assert(sizeof(CellRec) == 32, "CellRec must be one sector");

constexpr int32_t kFastBit = 1 << 30;  // PartLite::nb_flags: the CellRec points at the FP32 fast table
constexpr int kFastCShift = 24;        // bits 24..29: C/2 (C = 16-byte records per bucket incl. header, even)
constexpr int kFastListRecs = 6;  // records per fast list: header + edges, even (see the FP32 fast table below)
static_assert(kFastListRecs % 2 == 0 && kFastListRecs >= 2 && kFastListRecs <= 8, "fast list = 1..4 sectors");
constexpr int kFastMaxCount = 120;  // longest bucket list a fast part may have

struct __align__(32) EdgeRec {  // one L2 sector
    double sx, sy, ex, ey;
};

// The grid is defined on FINE cells; a coarse cell is a block of 2^rs x 2^rs fine cells (index >> rs), so the
// two levels nest exactly by construction.
struct GridParams {
    double x0, y0, x1, y1;  // union bbox of the valid parts (x0 > x1 when there is none)
    double inv_fw, inv_fh;  // fine cells per coordinate unit; 0 on a degenerate axis
    int32_t fgx, fgy;       // fine cells per axis = gx << rs, gy << rs
    int32_t gx, gy;         // coarse cells per axis
    int32_t rs;             // log2(fine cells per coarse cell and axis)
    int32_t wpr;            // raster words per fine row = ceil(fgx / 16): 2 bits per cell
};

}  // namespace gpl

struct gpl_pip_index {
    gpl_ctx *ctx = nullptr;
    const gpl_array *polys = nullptr;
    int64_t n_parts = 0, n_geoms = 0, n_buckets = 0, n_entries = 0, n_overflow = 0;
    gpl::GridParams grid;            // host copy, passed to the query kernel by value
    // one slab (so that a single L2 persisting access-policy window covers the whole index)
    uint8_t *slab = nullptr;
    size_t slab_bytes = 0;
    gpl::PartRec *parts = nullptr;
    gpl::CellRec *cells = nullptr;    // gx*gy
    int2 *cand01 = nullptr;           // gx*gy: polygon ROW of the cell's candidate #0 / #1 (-1 = none): raster codes 1 / 2
    uint2 *raster = nullptr;          // fgy rows x wpr words: x = 2 bits per fine cell (16 cells), y = row of the coarse cell's candidate #0
    int32_t *cell_overflow = nullptr; // ascending part ids of the cells' candidates
    int2 *bucket_range = nullptr;     // n_buckets: (start, end) into entries[]
    gpl::EdgeRec *entries = nullptr;
    int32_t *entry_ring = nullptr;    // ring index within part (0 = exterior), only if any part has holes
    float4 *fast = nullptr;           // FP32 fixed-stride bucket table of the plain parts (see "FP32 fast table" below)
    int64_t n_fast = 0;               // 16-byte records in `fast`
    size_t hot_bytes = 0;             // leading part of the slab the L2 persisting window covers (0 = all)
    bool multi = false;               // MULTIPOLYGON: parts[].geom differs from the part id
    bool any_holes = false;
    bool lean_ok = false;             // every valid part is a plain POLYGON with FP32 lists: LEAN walk
    int64_t n_not_fast = 0;           // valid parts without FP32 lists
    unsigned long long *n_deferred = nullptr;  // device counters inside the slab: [0] this launch, [1] since the build
    unsigned long long *phase_t = nullptr;     // 16 build-phase time stamps (ns), inside the slab
    uint32_t *deferred_list = nullptr;         // indices of deferred points (grown on demand)
    uint32_t deferred_cap = 0;
    int64_t bytes = 0;
};

namespace gpl {

// ------------------------------------------------------------------------------------------------
// monotone index functions (see the exactness argument at the top of the file)
// ------------------------------------------------------------------------------------------------
// fine cell of v: IEEE subtraction and multiplication by a non-negative constant are monotone, the conversion
// rounds towards -inf and saturates, min/max clamp: a monotone non-decreasing function of v.  NaN -> 0 (callers
// reject NaN first).  Build and query use THIS function, and the coarse cell is its value >> rs.
__device__ __forceinline__ int32_t fine_index(double v, double lo, double inv, int32_t n) {
    return min(max(__double2int_rd((v - lo) * inv), 0), n - 1);
}
// y-bucket of a part (float-valued parameters, double evaluation)
__device__ __forceinline__ int32_t mono_index(double v, double lo, double inv, int32_t n) {
    double t = floor((v - lo) * inv);
    // NaN never reaches here (callers reject points outside the closed bbox first)
    if (!(t > 0.0)) return 0;
    if (t >= (double)n) return n - 1;
    return (int32_t)t;
}
__device__ __forceinline__ int64_t ceil_div_dev(int64_t a, int64_t b) { return (a + b - 1) / b; }

// order-preserving encoding of doubles as unsigned integers (atomicMax on the union bbox)
__device__ __forceinline__ unsigned long long ord_enc(double d) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(d);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
__device__ __forceinline__ double ord_dec(unsigned long long u) {
    const unsigned long long b = (u >> 63) ? (u & 0x7fffffffffffffffULL) : ~u;
    return __longlong_as_double((long long)b);
}

// ------------------------------------------------------------------------------------------------
// index build: two cooperative kernels (count / fill) with one host round trip between them for the
// data-dependent sizes.  Round 1 issued ~27 small launches and two host syncs per build (0.35 ms, and the part of the
// step that scaled worst over 8 processes); the phases are the same, separated by grid barriers instead of launches.
// ------------------------------------------------------------------------------------------------
constexpr int kBuildThreads = 256;
constexpr int kMaxBuildCtas = 1024;
// edge slots per y-bucket x 100.  Round 1 (every point walks; kernel ms): 133: 2.18, 200: 2.03, 300: 1.95, 400: 1.98,
// 500: 2.07.  Round 2 (12 % of the points walk): 300: query 0.837 / build 0.54 ms, 600: query 0.842 / build 0.42 ms —
// half as many buckets to finish, the same query time.
constexpr int kSlotsX100 = 600;

enum {  // BuildArgs::acc slots (unsigned long long each, zeroed by the host before the count kernel)
    ACC_XMIN = 0, ACC_YMIN, ACC_XMAX, ACC_YMAX,  // union bbox, order-preserving encodings (min as max of the complement)
    ACC_HOLES, ACC_NOT_FAST, ACC_ITEMS, ACC_BUCKETS, ACC_ENTRIES, ACC_FAST, ACC_COUNT
};

struct BuildArgs {
    int type;
    int64_t P, n_geoms;
    const double2 *xy;
    const int64_t *geom_off, *part_off, *ring_off;
    const uint8_t *validity;
    int32_t G, rs;
    int64_t n_cells, NB_cap;
    // phase 1 (scratch)
    PartHeader *hdr;
    int32_t *nb;            // P: buckets per part; scanned in place into the chunk-local exclusive prefix
    int64_t *partial;       // 4 x kMaxBuildCtas chunk totals of the cooperative scans
    int32_t *cell_count;    // n_cells + 1
    int32_t *bcount;        // NB_cap + 1
    int2 *side_count;       // NB_cap + 1
    int32_t *fast_c, *fast_slots;  // P + 1
    int32_t *bucket_part;   // NB_cap + 1: the part that owns each y-bucket
    int2 *ovf_off;          // NB_cap + 1: first overflow record of the bucket's two FP32 lists, relative to the part's base
    unsigned long long *acc;
    GridParams *gp;
    // phase 2
    int64_t n_buckets, n_entries;
    int32_t *cell_cursor, *bcursor;
    int64_t *entry_edge;
    CellRec *cells;
    int2 *cand01;
    int32_t *items;
    PartRec *parts;
    int2 *bucket_range;
    EdgeRec *entries;
    int32_t *entry_ring;
    float4 *fast;
    uint2 *raster;          // per 16 fine cells: x = their 2-bit codes, y = the row of the coarse cell's candidate #0
    unsigned long long *n_deferred;
    unsigned long long *phase_t;  // 16 global-timer stamps (ns) taken by one thread at the phase boundaries of both kernels
};
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define GPL_STAMP(a, k)                                                              \
    do {                                                                             \
        if (blockIdx.x == 0 && threadIdx.x == 0 && (a).phase_t) (a).phase_t[k] = global_ns(); \
    } while (0)

__device__ __forceinline__ void part_rings(int type, int64_t part, const int64_t *geom_off, const int64_t *part_off,
                                           int64_t &r0, int64_t &r1) {
    if (type == GPL_POLYGON) {
        r0 = geom_off[part], r1 = geom_off[part + 1];
    } else {
        r0 = part_off[part], r1 = part_off[part + 1];
    }
}
// parent row of a part: POLYGON rows are their own part; MULTIPOLYGON: the row g with geom_off[g] <= p < geom_off[g+1]
__device__ __forceinline__ int32_t part_parent(const BuildArgs &a, int64_t p) {
    if (a.type == GPL_POLYGON) return (int32_t)p;
    int64_t lo = 0, hi = a.n_geoms;
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (a.geom_off[mid] <= p) lo = mid;
        else hi = mid;
    }
    return (int32_t)lo;
}

// exclusive scan of one value per thread across the CTA (kBuildThreads threads); `total` = CTA sum
__device__ __forceinline__ int64_t cta_scan_excl(int64_t v, int64_t &total, int64_t *sm /* kBuildThreads/32 + 1 */) {
    constexpr int NW = kBuildThreads / 32;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int64_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) sm[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const int64_t w = lane < NW ? sm[lane] : 0;
        int64_t winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < NW) sm[lane] = winc - w;
        if (lane == NW - 1) sm[NW] = winc;
    }
    __syncthreads();
    const int64_t excl = sm[wid] + inc - v;
    total = sm[NW];
    __syncthreads();  // the scratch is reused by the next call
    return excl;
}
// CTA-local exclusive scan of in[lo,hi) into out[lo,hi) (may alias); returns the chunk total in every thread
template <typename In, typename Out>
__device__ int64_t cta_chunk_scan(const In *in, Out *out, int64_t lo, int64_t hi, int64_t *sm) {
    int64_t carry = 0;
    for (int64_t base = lo; base < hi; base += kBuildThreads) {
        const int64_t i = base + threadIdx.x;
        const int64_t v = i < hi ? (int64_t)in[i] : 0;
        int64_t tot;
        const int64_t e = cta_scan_excl(v, tot, sm);
        if (i < hi) out[i] = (Out)(carry + e);
        carry += tot;
    }
    return carry;
}
// Cooperative scan, pass A: CTA b scans its chunk [b*L, (b+1)*L) locally and publishes the chunk total.
template <typename In, typename Out>
__device__ void grid_scan_local(const In *in, Out *out, int64_t n, int64_t *partial, int64_t *sm) {
    const int64_t L = ceil_div_dev(n > 0 ? n : 1, gridDim.x);
    const int64_t lo = min(n, (int64_t)blockIdx.x * L), hi = min(n, lo + L);
    const int64_t tot = cta_chunk_scan(in, out, lo, hi, sm);
    if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}
// pass B (after a grid barrier): exclusive prefix of the chunk totals in shared memory; returns the grand total
__device__ int64_t grid_scan_prefix(const int64_t *partial, int64_t *sm_prefix /* gridDim.x */, int64_t *sm) {
    const int64_t total = cta_chunk_scan(partial, sm_prefix, 0, (int64_t)gridDim.x, sm);
    __syncthreads();  // sm_prefix is read by every thread next
    return total;
}

// edge slot c of ring [c0,c1): (c -> c+1), or the implicit closing edge geo's Polygon::new would add
// for an open ring, or the degenerate edge of a 1-coordinate ring.  Returns false for "no edge".
__device__ __forceinline__ bool edge_of_slot(const double2 *__restrict__ xy, int64_t c, int64_t c0, int64_t c1, double2 &s,
                                             double2 &e) {
    s = xy[c];
    if (c + 1 < c1) {
        e = xy[c + 1];
        return true;
    }
    double2 first = xy[c0];
    if (c1 - c0 == 1) {
        e = s;
        return true;
    }
    if (first.x == s.x && first.y == s.y) return false;  // ring already closed
    e = first;
    return true;
}

// the x that separates the two one-sided edge lists of a part: the middle of its FLOAT x-range, formed the same
// way by the build (here) and by the query kernel (from PartLite)
__device__ __forceinline__ double fast_split_x(const PartHeader &h) {
    return 0.5 * ((double)__double2float_rd(h.xmin) + (double)__double2float_ru(h.xmax));
}
__device__ __forceinline__ PartLite lite_of(const PartHeader &h) {
    PartLite l;
    l.xminf = __double2float_rd(h.xmin);
    l.xmaxf = __double2float_ru(h.xmax);
    l.yminf = (float)h.by0;    // exact: by0 is a float value
    l.inv_hf = (float)h.inv_h;  // exact: inv_h is a float value
    l.nb_flags = (h.n_buckets & 0x00ffffff) | ((h.flags & 1) ? (int32_t)0x80000000 : 0);
    l.bucket_base = h.bucket_base;
    return l;
}
// the extent R the FP32 filter's error bounds are formed from — one expression, shared by the eligibility test of
// the build and by fast_walk
__device__ __forceinline__ float fast_extent(float xminf, float xmaxf, float inv_hf, int32_t nb) {
    const float height = inv_hf > 0.0f ? __fdividef((float)nb, inv_hf) : 0.0f;  // 2 ulp is plenty: R only feeds bounds with 2x slack
    return fmaxf(xmaxf - xminf, height);
}

__device__ __forceinline__ GridParams grid_from_acc(const BuildArgs &a) {
    GridParams g;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    if (a.acc[ACC_XMAX] == 0ULL) {  // no valid part: every point fails the bbox test
        g.x0 = g.y0 = inf, g.x1 = g.y1 = -inf;
    } else {
        g.x0 = ord_dec(~a.acc[ACC_XMIN]), g.y0 = ord_dec(~a.acc[ACC_YMIN]);
        g.x1 = ord_dec(a.acc[ACC_XMAX]), g.y1 = ord_dec(a.acc[ACC_YMAX]);
    }
    g.gx = g.gy = a.G, g.rs = a.rs;
    g.fgx = g.fgy = a.G << a.rs;
    g.wpr = (g.fgx + 15) >> 4;
    const double w = g.x1 - g.x0, h = g.y1 - g.y0;
    g.inv_fw = (w > 0.0 && isfinite(w)) ? (double)g.fgx / w : 0.0;
    g.inv_fh = (h > 0.0 && isfinite(h)) ? (double)g.fgy / h : 0.0;
    if (!isfinite(g.inv_fw)) g.inv_fw = 0.0;
    if (!isfinite(g.inv_fh)) g.inv_fh = 0.0;
    return g;
}

// ---- phase S0: per part bbox of the exterior ring, bucket count; union bbox ---------------------------------
__device__ void ph_headers(const BuildArgs &a, double *sm_box /* 4 x 8 */) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t warp = ((int64_t)blockIdx.x * kBuildThreads + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kBuildThreads) >> 5;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    double ux0 = inf, uy0 = inf, ux1 = -inf, uy1 = -inf;  // this warp's share of the union bbox
    bool holes_seen = false;
    for (int64_t p = warp; p < a.P; p += nwarps) {
        int64_t r0, r1;
        part_rings(a.type, p, a.geom_off, a.part_off, r0, r1);
        const int32_t g = part_parent(a, p);
        bool valid = bit_get(a.validity, g) && r1 > r0;
        double x0 = inf, y0 = inf, x1 = -inf, y1 = -inf;
        int64_t n_slots = 0;
        if (valid) {
            const int64_t c0 = a.ring_off[r0], c1 = a.ring_off[r0 + 1];
            if (c1 <= c0) valid = false;  // empty exterior: Outside for every point
            for (int64_t c = c0 + lane; c < c1; c += 32) {
                const double2 q = a.xy[c];
                x0 = fmin(x0, q.x), y0 = fmin(y0, q.y), x1 = fmax(x1, q.x), y1 = fmax(y1, q.y);
            }
            n_slots = a.ring_off[r1] - a.ring_off[r0];
        }
        x0 = warp_min(x0), y0 = warp_min(y0), x1 = warp_max(x1), y1 = warp_max(y1);
        if (!(x0 <= x1 && y0 <= y1)) valid = false;  // NaN-only exterior
        if (valid) {
            ux0 = fmin(ux0, x0), uy0 = fmin(uy0, y0), ux1 = fmax(ux1, x1), uy1 = fmax(uy1, y1);
            holes_seen = holes_seen || (r1 - r0 > 1);
        }
        if (lane == 0) {
            PartHeader h;
            h.xmin = x0, h.ymin = y0, h.xmax = x1, h.ymax = y1;
            // ~6 edge slots per y-bucket (kSlotsX100): on the config-2 stars a bucket lists ~9 of the 64 edges, and
            // each of its two one-sided lists (FP32 table) ~4.5.
            int64_t nb = valid ? (n_slots * 100 + kSlotsX100 - 1) / kSlotsX100 : 0;
            if (nb < 1) nb = valid ? 1 : 0;
            if (nb > 4096) nb = 4096;
            const float yminf = __double2float_rd(y0);
            const double by0 = (double)yminf;
            const double h_ext = y1 - by0;
            float inv_hf = (valid && h_ext > 0.0 && isfinite(h_ext)) ? __double2float_rn((double)nb / h_ext) : 0.0f;
            if (!isfinite(inv_hf)) inv_hf = 0.0f;
            h.by0 = by0;
            h.inv_h = (double)inv_hf;
            h.n_buckets = (int32_t)nb;
            h.bucket_base = 0;
            h.geom = g;
            h.flags = (valid ? 2 : 0) | ((r1 - r0 > 1) ? 1 : 0);
            a.hdr[p] = h;
            a.nb[p] = (int32_t)nb;
        }
    }
    // union bbox: warps -> CTA -> four atomics per CTA (same-address atomics serialise: one per part would cost more
    // than the whole build)
    if (lane == 0) sm_box[wid] = ux0, sm_box[8 + wid] = uy0, sm_box[16 + wid] = ux1, sm_box[24 + wid] = uy1;
    const bool any_h = __syncthreads_or(holes_seen);
    if (threadIdx.x == 0) {
        for (int w = 1; w < kBuildThreads / 32; ++w)
            ux0 = fmin(ux0, sm_box[w]), uy0 = fmin(uy0, sm_box[8 + w]), ux1 = fmax(ux1, sm_box[16 + w]), uy1 = fmax(uy1, sm_box[24 + w]);
        if (ux0 <= ux1 && uy0 <= uy1) {
            atomicMax(a.acc + ACC_XMIN, ~ord_enc(ux0));
            atomicMax(a.acc + ACC_YMIN, ~ord_enc(uy0));
            atomicMax(a.acc + ACC_XMAX, ord_enc(ux1));
            atomicMax(a.acc + ACC_YMAX, ord_enc(uy1));
        }
        if (any_h) a.acc[ACC_HOLES] = 1ULL;  // benign race: every writer stores the same value
    }
    __syncthreads();
}

// ---- coarse cells a part's bbox overlaps: pass 0 counts, pass 1 fills the per-cell candidate lists ---------------
template <int PASS>
__device__ void ph_cells(const BuildArgs &a, const GridParams &g) {
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    unsigned long long mine = 0;
    for (int64_t p = tid; p < a.P; p += nth) {
        const PartHeader h = a.hdr[p];
        if (!(h.flags & 2)) continue;
        const int32_t cx0 = fine_index(h.xmin, g.x0, g.inv_fw, g.fgx) >> g.rs, cx1 = fine_index(h.xmax, g.x0, g.inv_fw, g.fgx) >> g.rs;
        const int32_t cy0 = fine_index(h.ymin, g.y0, g.inv_fh, g.fgy) >> g.rs, cy1 = fine_index(h.ymax, g.y0, g.inv_fh, g.fgy) >> g.rs;
        for (int32_t cy = cy0; cy <= cy1; ++cy)
            for (int32_t cx = cx0; cx <= cx1; ++cx) {
                const int64_t c = (int64_t)cy * g.gx + cx;
                if (PASS == 0) {
                    atomicAdd(&a.cell_count[c], 1);
                    ++mine;
                } else {
                    const int32_t pos = atomicAdd(&a.cell_cursor[c], 1);
                    a.items[pos] = (int32_t)p;
                }
            }
    }
    if (PASS == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, o);
        if ((threadIdx.x & 31) == 0 && mine) atomicAdd(a.acc + ACC_ITEMS, mine);
    }
}

// ---- y-buckets: one warp per part; pass 0 counts bucket entries, pass 1 writes edge ids (global coord index) ------
template <int PASS>
__device__ void ph_buckets(const BuildArgs &a, const int64_t *sm_prefix, int64_t chunk_len) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * kBuildThreads + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kBuildThreads) >> 5;
    unsigned long long mine = 0;
    for (int64_t p = warp; p < a.P; p += nwarps) {
        PartHeader h = a.hdr[p];
        if (PASS == 0) {  // finish the scan of the bucket counts: chunk-local prefix + the prefix of the chunk totals
            h.bucket_base = a.nb[p] + (int32_t)sm_prefix[p / chunk_len];
            if (lane == 0) a.hdr[p].bucket_base = h.bucket_base;
        }
        if (!(h.flags & 2)) continue;
        const double xm = fast_split_x(h);
        int64_t r0, r1;
        part_rings(a.type, p, a.geom_off, a.part_off, r0, r1);
        for (int64_t r = r0; r < r1; ++r) {
            const int64_t c0 = a.ring_off[r], c1 = a.ring_off[r + 1];
            for (int64_t c = c0 + lane; c < c1; c += 32) {
                double2 s, e;
                if (!edge_of_slot(a.xy, c, c0, c1, s, e)) continue;
                // an edge with a NaN ordinate never satisfies geo's comparisons: it contributes nothing
                if (isnan(s.y) || isnan(e.y)) continue;
                const double ylo = fmin(s.y, e.y), yhi = fmax(s.y, e.y);
                // holes may stick out of the exterior's bbox: only the part of their y-range inside the
                // bucketed span [ymin,ymax] can hold a queried p.y (queries are bbox-filtered first)
                if (yhi < h.ymin || ylo > h.ymax) continue;
                const int32_t b0 = mono_index(fmax(ylo, h.ymin), h.by0, h.inv_h, h.n_buckets);
                const int32_t b1 = mono_index(fmin(yhi, h.ymax), h.by0, h.inv_h, h.n_buckets);
                for (int32_t b = b0; b <= b1; ++b) {
                    if (PASS == 0) {
                        atomicAdd(&a.bcount[h.bucket_base + b], 1);
                        ++mine;
                        // lengths of the two one-sided lists of the FP32 table (same predicate as ph_fast_fill)
                        if (fmax(s.x, e.x) >= xm) atomicAdd(&a.side_count[h.bucket_base + b].x, 1);
                        if (fmin(s.x, e.x) <= xm) atomicAdd(&a.side_count[h.bucket_base + b].y, 1);
                    } else {
                        const int32_t pos = atomicAdd(&a.bcursor[h.bucket_base + b], 1);
                        a.entry_edge[pos] = c;
                    }
                }
            }
        }
    }
    if (PASS == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, o);
        if (lane == 0 && mine) atomicAdd(a.acc + ACC_ENTRIES, mine);
    }
}

// ---- FP32 fast table --------------------------------------------------------------------------------
// The walk lives on L2: per point it pulls one cell sector plus its edge records, and it slows down as
// soon as the records it touches stop fitting in L2 next to the 1.6 GB point stream.  Plain parts (no holes,
// POLYGON rows) therefore get a second, denser table:
//   * edges as four FLOATS relative to the part origin O = (xminf, yminf): 16 bytes, two per sector;
//   * TWO lists per y-bucket ("sides").  A horizontal line through a spiky ring crosses many edges (12-17 on
//     the config-2 stars, whatever the bucket height), but only the crossings on ONE side of the point matter
//     to the winding number.  With xm = the middle of the part's float x-range (fast_split_x), a point with
//     p.x >= xm reads the list of edges with max(sx,ex) >= xm (the others lie strictly left of it: they neither
//     cross the rightward ray nor contain p); a point with p.x < xm reads the list of edges with
//     min(sx,ex) <= xm stored MIRRORED in x (x' = xmaxf - x): mirroring turns "left of p" into "right of p'"
//     and negates the winding number, and only wn != 0 is consumed;
//   * fixed stride: list (b, side) of a part starts at fast_base + (2b + side) * kFastListRecs records: one
//     header {count, overflow offset} + kFastListRecs-1 edge slots, unused slots hold an inert sentinel (+inf
//     ordinates) — no (start,end) lookup, the whole list is one batch of 256-bit loads.  Longer lists
//     continue in a per-part overflow area addressed from the header (exactly sized: ph_buckets counts both
//     sides).
// The floats only feed a FILTER with a rigorous error bound (fast_edge_rule); anything it cannot certify is
// re-evaluated from the f64 records by the exact kernel.  kFastBit lives in PartLite::nb_flags.

// per part: eligibility and its number of 16-byte records (main lists + overflow)
__device__ void ph_fast_plan(const BuildArgs &a) {
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    unsigned long long slots_sum = 0, not_fast = 0;
    for (int64_t p = tid; p < a.P; p += nth) {
        const PartHeader h = a.hdr[p];
        int32_t c = 0, slots = 0;
        for (int32_t b = 0; b < h.n_buckets; ++b) a.bucket_part[h.bucket_base + b] = (int32_t)p;
        if (a.type == GPL_POLYGON && (h.flags & 2) && !(h.flags & 1)) {
            int32_t mx = 0, ovf = 0;
            const int32_t ovf0 = h.n_buckets * 2 * kFastListRecs;  // the overflow area follows the fixed-stride lists
            for (int32_t b = 0; b < h.n_buckets; ++b) {
                mx = max(mx, a.bcount[h.bucket_base + b]);
                const int2 sc = a.side_count[h.bucket_base + b];
                const int32_t o0 = (max(sc.x - (kFastListRecs - 1), 0) + 1) & ~1, o1 = (max(sc.y - (kFastListRecs - 1), 0) + 1) & ~1;
                a.ovf_off[h.bucket_base + b] = make_int2(ovf0 + ovf, ovf0 + ovf + o0);
                ovf += o0 + o1;
            }
            // The filter's bounds eta = 2^-20 R and B ~ 2^-16 R^2 are formed in FLOAT: they must neither underflow
            // (R^2 subnormal: the relative-error argument of fast_edge_rule no longer holds) nor overflow (B = inf
            // defers every point).  Parts outside 2^-50 <= R <= 2^50 keep the f64 walk.
            const PartLite l = lite_of(h);
            const float R = fast_extent(l.xminf, l.xmaxf, l.inv_hf, h.n_buckets);
            const bool scale_ok = R >= 8.8817841970012523e-16f && R <= 1.125899906842624e15f;
            if (mx <= kFastMaxCount && scale_ok) {
                c = kFastListRecs;
                slots = h.n_buckets * 2 * kFastListRecs + ovf;
            }
        }
        if ((h.flags & 2) && c == 0) ++not_fast;  // a valid part the FP32 table cannot hold
        a.fast_c[p] = c;
        a.fast_slots[p] = slots;
        slots_sum += (unsigned long long)slots;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        slots_sum += __shfl_down_sync(0xffffffffu, slots_sum, o);
        not_fast += __shfl_down_sync(0xffffffffu, not_fast, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (slots_sum) atomicAdd(a.acc + ACC_FAST, slots_sum);
        if (not_fast) atomicAdd(a.acc + ACC_NOT_FAST, not_fast);
    }
}
// One THREAD per y-bucket finishes it: orders the bucket's edge ids where a consumer needs it (parts with holes),
// materialises the 32-byte f64 records (+ ring index when holes exist) and writes the bucket's two FP32 lists (header, float
// edges relative to the part origin, sentinels, overflow records).  Round 2's first build did these as three warp-per-part
// phases separated by grid barriers; a part's ~22 buckets then cost ~44 dependent L2 round trips per warp.  Here every
// load of a bucket (edge ids, coordinates) is independent of the others and 227 k buckets run side by side.
__device__ void ph_bucket_finish(const BuildArgs &a, const int32_t *__restrict__ bstart) {
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    const float inf = __int_as_float(0x7f800000);
    const float4 sentinel = make_float4(0.0f, inf, 0.0f, inf);  // inert: +inf ordinates never straddle a finite p.y
    for (int64_t gb = tid; gb < a.n_buckets; gb += nth) {
        const int32_t e0 = bstart[gb], n = bstart[gb + 1] - e0;
        const int32_t p = a.bucket_part[gb];
        const PartHeader h = a.hdr[p];
        int64_t r0, r1;
        part_rings(a.type, p, a.geom_off, a.part_off, r0, r1);
        // ---- order: parts WITH holes need their entries grouped by ring (ascending edge id does it: the bucket walk switches
        // ring when the ring index changes).  For a hole-free part the order in which the atomic cursors filled the bucket is
        // irrelevant to every consumer (winding sums and the two one-sided lists are order-independent), so it is kept.
        if (h.flags & 1) {
            int64_t *g = a.entry_edge + e0;
            for (int32_t i = 1; i < n; ++i) {
                const int64_t v = g[i];
                int32_t j = i - 1;
                while (j >= 0 && g[j] > v) {
                    g[j + 1] = g[j];
                    --j;
                }
                g[j + 1] = v;
            }
        }
        // ---- FP32 lists of this bucket (plain parts only)
        const bool fast = a.fast_c[p] > 0;
        const int32_t b = (int32_t)(gb - h.bucket_base);
        float4 *base = nullptr, *list0 = nullptr, *list1 = nullptr;
        int2 ovf = make_int2(0, 0);
        double ox = 0.0, mx = 0.0, oy = 0.0, xm = 0.0;
        if (fast) {
            base = a.fast + (int64_t)a.fast_slots[p];
            list0 = base + ((int64_t)b * 2) * kFastListRecs, list1 = list0 + kFastListRecs;
            ovf = a.ovf_off[gb];
            ox = (double)__double2float_rd(h.xmin), mx = (double)__double2float_ru(h.xmax), oy = h.by0;
            xm = fast_split_x(h);  // == 0.5 * (ox + mx); the query kernel forms it from PartLite
        }
        int32_t c0 = 0, c1 = 0;  // lengths of the two one-sided lists
        const int64_t ext0 = a.ring_off[r0], ext1 = a.ring_off[r0 + 1];
        // four entries at a time: their edge ids, then their coordinates, are loaded together (read-only path) before
        // anything is stored — one entry per iteration cost two dependent L2 round trips each
        for (int32_t k0 = 0; k0 < n; k0 += 4) {
            const int32_t mm = min(4, n - k0);
            int64_t cc[4], rr[4];
            double2 ss[4], ee[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) cc[j] = j < mm ? __ldg(a.entry_edge + e0 + k0 + j) : ext0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int64_t r = r0, rc0 = ext0, rc1 = ext1;
                if (h.flags & 1) {  // ring of coordinate c: rings of a part are few; linear search from the exterior
                    while (r + 1 < r1 && a.ring_off[r + 1] <= cc[j]) ++r;
                    rc0 = a.ring_off[r], rc1 = a.ring_off[r + 1];
                }
                rr[j] = r - r0;
                // edge_of_slot on the read-only path: (c -> c+1), or the closing edge back to the ring's first coordinate,
                // or the degenerate edge of a 1-coordinate ring (entries never name a "no edge" slot)
                ss[j] = __ldg(a.xy + cc[j]);
                ee[j] = cc[j] + 1 < rc1 ? __ldg(a.xy + cc[j] + 1) : (rc1 - rc0 == 1 ? ss[j] : __ldg(a.xy + rc0));
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (j >= mm) break;
                const double2 s = ss[j], e = ee[j];
                const int32_t k = k0 + j;
                EdgeRec rec;
                rec.sx = s.x, rec.sy = s.y, rec.ex = e.x, rec.ey = e.y;
                a.entries[e0 + k] = rec;
                if (a.entry_ring) a.entry_ring[e0 + k] = (int32_t)rr[j];
                if (fast) {
                    if (fmax(s.x, e.x) >= xm) {  // right-hand list: coordinates relative to (xminf, yminf)
                        const float4 f = make_float4(__double2float_rn(s.x - ox), __double2float_rn(s.y - oy), __double2float_rn(e.x - ox),
                                                     __double2float_rn(e.y - oy));
                        if (c0 < kFastListRecs - 1) list0[1 + c0] = f;
                        else base[ovf.x + c0 - (kFastListRecs - 1)] = f;
                        ++c0;
                    }
                    if (fmin(s.x, e.x) <= xm) {  // left-hand list, mirrored in x
                        const float4 f = make_float4(__double2float_rn(mx - s.x), __double2float_rn(s.y - oy), __double2float_rn(mx - e.x),
                                                     __double2float_rn(e.y - oy));
                        if (c1 < kFastListRecs - 1) list1[1 + c1] = f;
                        else base[ovf.y + c1 - (kFastListRecs - 1)] = f;
                        ++c1;
                    }
                }
            }
        }
        if (fast) {
            for (int32_t k = c0; k < kFastListRecs - 1; ++k) list0[1 + k] = sentinel;
            for (int32_t k = c1; k < kFastListRecs - 1; ++k) list1[1 + k] = sentinel;
            const int32_t n0 = max(c0 - (kFastListRecs - 1), 0), n1 = max(c1 - (kFastListRecs - 1), 0);
            list0[0] = make_float4(__int_as_float(c0), __int_as_float(n0 ? ovf.x : 0), 0.0f, 0.0f);
            list1[0] = make_float4(__int_as_float(c1), __int_as_float(n1 ? ovf.y : 0), 0.0f, 0.0f);
            if (n0 & 1) base[ovf.x + n0] = sentinel;  // overflow runs are padded to an even number of records
            if (n1 & 1) base[ovf.y + n1] = sentinel;
        }
    }
}

// one thread per segment: insertion sort (lists are a handful of items) — makes cell candidate lists
// ascending by part id and bucket lists ascending by edge id (=> grouped by ring, deterministic).
template <typename T>
__device__ void ph_sort_segments(T *__restrict__ items, const int32_t *__restrict__ seg_start, int64_t n_seg) {
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    for (int64_t s = tid; s < n_seg; s += nth) {
        const int32_t a = seg_start[s], b = seg_start[s + 1];
        for (int32_t i = a + 1; i < b; ++i) {
            const T v = items[i];
            int32_t j = i - 1;
            while (j >= a && items[j] > v) {
                items[j + 1] = items[j];
                --j;
            }
            items[j + 1] = v;
        }
    }
}

// the one-sector record of every coarse cell + the rows of its first two candidates (raster codes 1 / 2)
__device__ void ph_cell_finish(const BuildArgs &a, const int32_t *__restrict__ cell_start) {
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    for (int64_t c = tid; c < a.n_cells; c += nth) {
        const int32_t s = cell_start[c], e = cell_start[c + 1];
        CellRec r;
        r.count = e - s;
        r.first = (e - s == 1) ? a.items[s] : s;
        int2 cand = make_int2(-1, -1);
        if (e > s) {
            const int32_t p0 = a.items[s];
            r.lite = lite_of(a.hdr[p0]);
            if (e - s == 1 && a.fast_c[p0] > 0) {  // the one-load fast path: parameters of the FP32 table
                r.lite.nb_flags |= kFastBit | ((kFastListRecs / 2) << kFastCShift);
                r.lite.bucket_base = a.fast_slots[p0];
            }
            cand.x = a.hdr[p0].geom;
            if (e - s > 1) cand.y = a.hdr[a.items[s + 1]].geom;
        } else {
            r.lite.xminf = r.lite.xmaxf = r.lite.yminf = r.lite.inv_hf = 0.0f;
            r.lite.nb_flags = r.lite.bucket_base = 0;
        }
        a.cells[c] = r;
        a.cand01[c] = cand;
    }
}
// the row of candidate #0 next to the codes it qualifies: raster code 1 (36 % of config 2's points) then needs no second
// gather.  A word (16 fine cells) lies inside one coarse cell when 2^rs >= 16; otherwise the word keeps -2 = "ask cand01".
__device__ void ph_raster_cand(const BuildArgs &a, const GridParams &g) {
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    const int64_t n_words = (int64_t)g.fgy * g.wpr;
    for (int64_t i = tid; i < n_words; i += nth) {
        const int32_t fy = (int32_t)(i / g.wpr), wx = (int32_t)(i - (int64_t)fy * g.wpr);
        uint32_t v = 0xfffffffeu;
        if (g.rs >= 4) v = (uint32_t)a.cand01[(int64_t)(fy >> g.rs) * g.gx + ((wx << 4) >> g.rs)].x;
        a.raster[i].y = v;
    }
}
__device__ void ph_part_recs(const BuildArgs &a) {
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    for (int64_t p = tid; p < a.P; p += nth) {
        const PartHeader h = a.hdr[p];
        PartRec r;
        r.lite = lite_of(h);  // bucket_base: the f64 bucket table (general path, exact kernel)
        r.geom = h.geom;
        r.pad = 0;
        if (a.fast_c[p] > 0) {  // the FP32 lists of this part, for candidates read through the PartRec (LEAN walk)
            r.lite.nb_flags |= kFastBit | ((kFastListRecs / 2) << kFastCShift);
            r.pad = a.fast_slots[p];
        }
        a.parts[p] = r;
    }
}
// ------------------------------------------------------------------------------------------------
// exact rule (shared by the raster classification, the deferred kernel and the pair mode)
// ------------------------------------------------------------------------------------------------
// geo's coord_pos_relative_to_ring step with the full adaptive predicate (exact sign always)
__device__ __forceinline__ void edge_rule_exact(double sx, double sy, double ex, double ey, double px, double py, int &wn,
                                                bool &boundary) {
    if (sy <= py) {
        if (ey >= py) {
            double o = orient2d(sx, sy, ex, ey, px, py);
            if (o > 0.0 && ey != py) wn += 1;
            else if (o == 0.0 && value_in_between(px, sx, ex)) boundary = true;
        }
    } else if (ey <= py) {
        double o = orient2d(sx, sy, ex, ey, px, py);
        if (o < 0.0) wn -= 1;
        else if (o == 0.0 && value_in_between(px, sx, ex)) boundary = true;
    }
}

// Polygon::contains(coord) over the entries [e0,e1) of one bucket, serial and exact: used for parts
// with holes and for the (rare) points the fast filter could not decide.
// No holes: Inside <=> not on any listed edge and winding != 0.
// Holes: entries are grouped by ring (ascending); exterior must wind, every hole must not, and no
// ring may have p on its boundary (geo: boundary of exterior or of a hole => not Inside).
static __device__ __noinline__ bool bucket_contains_exact(const EdgeRec *__restrict__ entries,
                                                          const int32_t *__restrict__ entry_ring, bool holes, int32_t e0, int32_t e1,
                                                          double px, double py) {
    int wn = 0;
    bool boundary = false;
    if (e0 == e1) return false;
    int32_t cur = holes ? entry_ring[e0] : 0;
    if (cur != 0) return false;  // no exterior edge near p.y: winding 0 => Outside
    bool ok = true;
    for (int32_t k = e0; k < e1; ++k) {
        if (holes) {
            int32_t ring = entry_ring[k];
            if (ring != cur) {
                ok = ok && (cur == 0 ? (wn != 0) : (wn == 0));
                cur = ring;
                wn = 0;
            }
        }
        EdgeRec ed = entries[k];
        edge_rule_exact(ed.sx, ed.sy, ed.ex, ed.ey, px, py, wn, boundary);
    }
    ok = ok && (cur == 0 ? (wn != 0) : (wn == 0));
    return ok && !boundary;
}

// ------------------------------------------------------------------------------------------------
// raster: 2 bits per fine cell
// ------------------------------------------------------------------------------------------------
// Codes: 0 = outside every part; 1 / 2 = strictly inside candidate #0 / #1 of the coarse cell (its ascending
// part list) and outside every other part; 3 = walk.  All writes are atomicOr, so codes compose: a second
// "inside" from another part turns 1|2 into 3, a boundary mark turns anything into 3.
//
// Why a code other than 3 is exact.  Work in cell units: T(v) = (v - lo) * inv as a REAL map; the computed
// (v - lo) * inv of a double differs from T(v) by at most 2^-31 cells (two roundings of 2^-53 relative, at most
// 2^20 fine cells per axis), so every double that maps to cell (c, r) lies in the real rectangle
// Q(c,r) = T^-1([c - e/2, c + 1 + e/2] x [r - e/2, r + 1 + e/2]) with e = 1e-6.  raster_mark_row marks every cell
// whose e-inflated square meets the segment (row by row, with the slack analysed there), for every ring segment of
// every valid part — including the closing segment geo's Polygon::new adds and 1-coordinate rings.  A cell that is
// not marked by part P therefore has no point of P's rings in Q(c,r): Q is convex, so it lies in one face of each
// ring's arrangement, every winding number geo computes is constant on it and no point of it is on a boundary;
// horizontally adjacent unmarked cells overlap (their Q's share a strip) and lie in the same face.  One exact
// evaluation of geo's rule at one representative double that maps to the cell classifies every query point that maps
// to it.  Anything this argument does not cover (degenerate axis, a representative that does not map back, non-finite
// coordinates, more than two containing candidates) is coded 3.
__device__ __forceinline__ void raster_or_span(uint2 *__restrict__ raster, int32_t wpr, int32_t fy, int32_t c0, int32_t c1,
                                               uint32_t code) {
    uint2 *row = raster + (int64_t)fy * wpr;
    const uint32_t rep = code * 0x55555555u;
    for (int32_t w = c0 >> 4; w <= (c1 >> 4); ++w) {
        const int32_t lo = max(c0 - (w << 4), 0), hi = min(c1 - (w << 4), 15);  // inclusive cell range inside word w
        const uint32_t m = (0xffffffffu >> (2 * (15 - hi))) & (0xffffffffu << (2 * lo));
        atomicOr(&row[w].x, rep & m);
    }
}
// One row of the marking: code 3 for every fine cell of row r within 1e-6 cells of the segment whose images in cell units
// are (tsx,tsy)-(tex,tey).  inv_dy = 1 / (tey - tsy), or 0 for a segment that is nearly horizontal in cell units.
__device__ __forceinline__ void raster_mark_row(uint2 *__restrict__ raster, const GridParams &g, int32_t r, double tsx, double tsy,
                                                double tex, double tey, double inv_dy) {
    const double eps = 1e-6;
    double xa, xb;
    if (inv_dy == 0.0) {  // |dy| < 1e-3 cells: the whole x-range on each of the (at most 3) rows
        xa = fmin(tsx, tex), xb = fmax(tsx, tex);
    } else {
        // parameter range of the segment inside the slab [r - eps, r + 1 + eps].  Errors: the endpoints are within
        // 2^-30 of their true images and so is dy, i.e. lambda is off by at most 4 * 2^-30 / |dy| — 270 times
        // smaller than the eps / |dy| the slab was widened by; x(lambda) adds a few 2^-32.  The 2e-6 margin below
        // covers the rest (and the 2^-52 relative error of multiplying by the reciprocal instead of dividing).
        double l0 = ((double)r - eps - tsy) * inv_dy, l1 = ((double)r + 1.0 + eps - tsy) * inv_dy;
        if (l0 > l1) {
            const double t = l0;
            l0 = l1, l1 = t;
        }
        l0 = fmax(l0, 0.0), l1 = fmin(l1, 1.0);
        if (l0 > l1) return;  // a clamped border row the segment does not reach (no query point maps there)
        const double dx = tex - tsx;
        xa = tsx + l0 * dx, xb = tsx + l1 * dx;
        if (xa > xb) {
            const double t = xa;
            xa = xb, xb = t;
        }
    }
    const int32_t c0 = min(max(__double2int_rd(xa - 2e-6), 0), g.fgx - 1), c1 = min(max(__double2int_rd(xb + 2e-6), 0), g.fgx - 1);
    raster_or_span(raster, g.wpr, r, c0, c1, 3u);
}
// raster code of "strictly inside part `part` only" in coarse cell (cx, cy): 1 / 2 for candidate #0 / #1, else 3
__device__ __forceinline__ uint32_t raster_rank_code(const BuildArgs &a, const GridParams &g, const int32_t *__restrict__ cell_start,
                                                     int32_t cx, int32_t cy, int32_t part) {
    const int64_t c = (int64_t)cy * g.gx + cx;
    const int32_t s = cell_start[c], e = cell_start[c + 1];
    if (s < e && a.items[s] == part) return 1u;
    if (s + 1 < e && a.items[s + 1] == part) return 2u;
    return 3u;
}
// OR the inside code of `part` over cells [lo, hi] of fine row fy (the code depends on the coarse column).
// `codes` (or nullptr): the part's codes in the coarse cells of its bbox, row-major from (cx0, cy0), ncx per row — the two
// dependent global loads of raster_rank_code per span were the latency of the whole phase.
__device__ __forceinline__ void raster_fill_span(const BuildArgs &a, const GridParams &g, const int32_t *__restrict__ cell_start,
                                                 int32_t fy, int32_t lo, int32_t hi, int32_t part, const uint8_t *codes, int32_t cx0,
                                                 int32_t cy0, int32_t ncx) {
    for (int32_t cc = lo >> g.rs; cc <= (hi >> g.rs); ++cc) {
        const int32_t x0 = max(lo, cc << g.rs), x1 = min(hi, ((cc + 1) << g.rs) - 1);
        const uint32_t code = codes ? (uint32_t)codes[((fy >> g.rs) - cy0) * ncx + (cc - cx0)] : raster_rank_code(a, g, cell_start, cc, fy >> g.rs, part);
        raster_or_span(a.raster, g.wpr, fy, x0, x1, code);
    }
}

// The raster of one part, built by one warp in chunks of 32 fine rows of the part's bbox:
//   edge-major: every lane takes edges of the part's rings; for every row of the chunk an edge comes near, it marks the
//               cells along the edge (code 3) and, when the edge straddles the row's CENTRE LINE y = ry (geo's half-open
//               rule: upward s.y <= ry < e.y, downward e.y <= ry < s.y), records the crossing cell, direction and ring
//               in the row's list in shared memory;
//   row-major : every lane takes one row, sorts its crossings by cell and ORs the inside code over the cells strictly
//               between consecutive crossings whose winding numbers say Inside (exterior ring winds, no hole winds).
// Why this is exact for every cell that keeps a code other than 3: such a cell is not marked, so (argument above) one
// representative decides it — take the cell centre (c + 1/2, ry).  geo's winding number of a ring at that point counts the
// ring's upward edges the point is left of minus the downward edges it is right of, i.e. the straddling edges whose crossing
// with y = ry lies at larger x.  The true crossing and the computed one (lambda is off by < 2^-29 / |dy|, far less than
// the half slab height the marks cover) both lie in the contiguous run of cells this edge marked on this row; an unmarked
// cell is outside that run, hence on the same side of both: comparing CELL indices orders the centre and the crossing
// exactly.  Everything the lists cannot hold (more than kRowCross crossings in a row, a row whose centre does not map
// back to it) is coded 3 over the part's whole column range, which is always safe.
constexpr int kRowCross = 24;  // a horizontal line through a config-2 star crosses 12-17 edges
constexpr int kRasterCodeCells = 64;  // coarse cells of a part's bbox whose codes are staged (a config-2 part covers 4-9)
constexpr int kRowStride = kRowCross + 1;  // odd stride: the 32 lists of a chunk do not collide on banks
struct RasterSmem {
    double ry[kBuildThreads / 32][32];  // centre-line ordinate of every row of the chunk (one division per row, not per edge)
    int32_t cnt[kBuildThreads / 32][32];
    uint32_t list[kBuildThreads / 32][32 * kRowStride];  // cell (20 bits) | down (bit 20) | ring (bits 21..31, saturated)
    uint8_t code[kBuildThreads / 32][kRasterCodeCells];   // the part's inside code in every coarse cell of its bbox
};
__device__ void ph_raster(const BuildArgs &a, const GridParams &g, const int32_t *__restrict__ cell_start, RasterSmem &sm) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t warp = ((int64_t)blockIdx.x * kBuildThreads + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kBuildThreads) >> 5;
    if (g.inv_fw == 0.0 || g.inv_fh == 0.0) return;  // degenerate axis: the raster was filled with 3 (fill kernel, T0)
    int32_t *cnt = sm.cnt[wid];
    uint32_t *list = sm.list[wid];
    double *row_y = sm.ry[wid];
    // work item = (part, k): the chunks ra = fy0 + 32 (k + K j) of the part.  A part's bbox is about one coarse cell high,
    // i.e. K = 2^rs / 32 chunks; they are independent (every raster write is an atomicOr), so config 4's 1 000 parts keep
    // 4 000 warps busy instead of 1 000.
    const int32_t K = max(1, min(8, (1 << g.rs) >> 5));
    for (int64_t it = warp; it < a.P * K; it += nwarps) {
        const int64_t p = it / K;
        const int32_t kk = (int32_t)(it - p * K);
        const PartHeader h = a.hdr[p];
        if (!(h.flags & 2)) continue;
        int64_t r0, r1;
        part_rings(a.type, p, a.geom_off, a.part_off, r0, r1);
        const int32_t fx0 = fine_index(h.xmin, g.x0, g.inv_fw, g.fgx), fx1 = fine_index(h.xmax, g.x0, g.inv_fw, g.fgx);
        const int32_t fy0 = fine_index(h.ymin, g.y0, g.inv_fh, g.fgy), fy1 = fine_index(h.ymax, g.y0, g.inv_fh, g.fgy);
        bool irregular = false;
        // the part's inside code per coarse cell of its bbox, once per part
        const int32_t cx0 = fx0 >> g.rs, cy0 = fy0 >> g.rs, ncx = (fx1 >> g.rs) - cx0 + 1, ncy = (fy1 >> g.rs) - cy0 + 1;
        const bool staged = (int64_t)ncx * ncy <= kRasterCodeCells;
        const uint8_t *codes = staged ? sm.code[wid] : nullptr;
        __syncwarp();  // the previous part's rows are done with the table
        if (staged)
            for (int32_t k = lane; k < ncx * ncy; k += 32)
                sm.code[wid][k] = (uint8_t)raster_rank_code(a, g, cell_start, cx0 + k % ncx, cy0 + k / ncx, (int32_t)p);
        __syncwarp();
        for (int32_t ra = fy0 + 32 * kk; ra <= fy1; ra += 32 * K) {
            const int32_t rb = min(ra + 31, fy1);
            cnt[lane] = 0;
            row_y[lane] = g.y0 + ((double)(ra + lane) + 0.5) / g.inv_fh;
            __syncwarp();
            // ---- edge-major: marks + centre-line crossings of the rows [ra, rb]
            for (int64_t r = r0; r < r1; ++r) {
                const int64_t c0 = a.ring_off[r], c1 = a.ring_off[r + 1];
                const uint32_t ring_tag = (uint32_t)((r - r0) < 2047 ? (r - r0) : 2047) << 21;
                for (int64_t c = c0 + lane; c < c1; c += 32) {
                    double2 s, e;
                    if (!edge_of_slot(a.xy, c, c0, c1, s, e)) continue;
                    // an edge with a NaN coordinate never satisfies geo's comparisons (NaN ordinate) or never yields a
                    // non-zero / zero orientation (NaN abscissa): it contributes nothing and bounds no face
                    if (isnan(s.x) || isnan(s.y) || isnan(e.x) || isnan(e.y)) continue;
                    // the arguments of fine_index, as the query kernel computes them
                    const double tsx = (s.x - g.x0) * g.inv_fw, tsy = (s.y - g.y0) * g.inv_fh;
                    const double tex = (e.x - g.x0) * g.inv_fw, tey = (e.y - g.y0) * g.inv_fh;
                    if (!(isfinite(tsx) && isfinite(tsy) && isfinite(tex) && isfinite(tey))) {
                        irregular = true;
                        continue;
                    }
                    const double ylo = fmin(tsy, tey), yhi = fmax(tsy, tey);
                    const int32_t er0 = max(min(max(__double2int_rd(ylo - 1e-6), 0), g.fgy - 1), ra);
                    const int32_t er1 = min(min(max(__double2int_rd(yhi + 1e-6), 0), g.fgy - 1), rb);
                    const double tdy = tey - tsy, tdx = tex - tsx;
                    const double inv_dy = fabs(tdy) < 1e-3 ? 0.0 : 1.0 / tdy;  // one division per edge and chunk
                    for (int32_t row = er0; row <= er1; ++row) {
                        raster_mark_row(a.raster, g, row, tsx, tsy, tex, tey, inv_dy);
                        const double ry = row_y[row - ra];
                        const bool up = s.y <= ry && e.y > ry, down = s.y > ry && e.y <= ry;
                        if (up || down) {
                            // crossing with the centre line, in cell units: its ordinate there is row + 1/2 up to 2^-31; only the
                            // cell is used, and any lambda inside the slab lands in the run of cells this edge marks on this row
                            double lam = inv_dy != 0.0 ? ((double)row + 0.5 - tsy) * inv_dy : 0.5;
                            lam = fmin(fmax(lam, 0.0), 1.0);
                            const int32_t cj = min(max(__double2int_rd(tsx + lam * tdx), 0), g.fgx - 1);
                            const int32_t slot = atomicAdd(&cnt[row - ra], 1);
                            if (slot < kRowCross) list[(row - ra) * kRowStride + slot] = (uint32_t)cj | (down ? (1u << 20) : 0u) | ring_tag;
                        }
                    }
                }
            }
            __syncwarp();
            // ---- row-major: one lane per row of the chunk
            const int32_t fy = ra + lane;
            if (fy <= rb) {
                const int32_t n = cnt[lane];
                const double ry = row_y[lane];
                uint32_t *L = list + lane * kRowStride;
                if (n > kRowCross || fine_index(ry, g.y0, g.inv_fh, g.fgy) != fy) {
                    raster_or_span(a.raster, g.wpr, fy, fx0, fx1, 3u);  // cannot be classified from the list: walk
                } else if (n > 0) {
                    for (int i = 1; i < n; ++i) {  // insertion sort by cell (the low 20 bits)
                        const uint32_t v = L[i];
                        int j = i - 1;
                        while (j >= 0 && (L[j] & 0xfffffu) > (v & 0xfffffu)) {
                            L[j + 1] = L[j];
                            --j;
                        }
                        L[j + 1] = v;
                    }
                    if (r1 - r0 == 1) {
                        // a part without holes: the winding number of interval k is the sum of the directions of entries k..n-1 —
                        // a running sum from the right (the general loop below recomputes it per interval: O(n^2) per row, and a
                        // config-2 star has 12-17 crossings per row)
                        int wn = 0;
                        for (int k = n - 1; k >= 1; --k) {
                            wn += (L[k] & (1u << 20)) ? -1 : 1;
                            const int32_t lo = (int32_t)(L[k - 1] & 0xfffffu) + 1, hi = (int32_t)(L[k] & 0xfffffu) - 1;
                            if (lo <= hi && wn != 0) raster_fill_span(a, g, cell_start, fy, lo, hi, (int32_t)p, codes, cx0, cy0, ncx);
                        }
                    } else
                    for (int k = 1; k < n; ++k) {  // cells strictly between crossing k-1 and crossing k
                        const int32_t lo = (int32_t)(L[k - 1] & 0xfffffu) + 1, hi = (int32_t)(L[k] & 0xfffffu) - 1;
                        if (lo > hi) continue;
                        // winding numbers at the interval = crossings to its right (entries k..n-1), ring by ring
                        int wn_ext = 0;
                        bool in_hole = false;
                        for (int j = k; j < n; ++j) {
                            const uint32_t ring = L[j] >> 21;
                            const int dir = (L[j] & (1u << 20)) ? -1 : 1;
                            if (ring == 0u) {
                                wn_ext += dir;
                            } else {
                                bool first = true;  // sum this hole once, at its first entry
                                for (int i = k; i < j; ++i) first = first && (L[i] >> 21) != ring;
                                if (first) {
                                    int w = 0;
                                    for (int i = j; i < n; ++i) w += ((L[i] >> 21) == ring) ? ((L[i] & (1u << 20)) ? -1 : 1) : 0;
                                    in_hole = in_hole || w != 0;
                                }
                            }
                        }
                        // ring indices saturate at 2047: a part with more rings cannot separate its holes — walk
                        bool saturated = false;
                        for (int j = k; j < n; ++j) saturated = saturated || (L[j] >> 21) == 2047u;
                        if (saturated) raster_or_span(a.raster, g.wpr, fy, lo, hi, 3u);
                        else if (wn_ext != 0 && !in_hole) raster_fill_span(a, g, cell_start, fy, lo, hi, (int32_t)p, codes, cx0, cy0, ncx);
                    }
                }
            }
            __syncwarp();
        }
        if (__any_sync(0xffffffffu, irregular)) {  // infinite coordinates: every cell of the grid takes the walk
            for (int32_t fy = lane; fy < g.fgy; fy += 32) raster_or_span(a.raster, g.wpr, fy, 0, g.fgx - 1, 3u);
        }
    }
}

// ---- the two cooperative kernels --------------------------------------------------------------------------
__global__ void __launch_bounds__(kBuildThreads) k_pip_build_count(const BuildArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ int64_t sm_scan[kBuildThreads / 32 + 1];
    __shared__ int64_t sm_prefix[kMaxBuildCtas];
    __shared__ double sm_box[32];
    __shared__ GridParams sm_g;
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    // S0: zero the counters the later phases add into; headers + union bbox
    GPL_STAMP(a, 0);
    for (int64_t i = tid; i <= a.n_cells; i += nth) a.cell_count[i] = 0;
    for (int64_t i = tid; i <= a.NB_cap; i += nth) {
        a.bcount[i] = 0;
        a.side_count[i] = make_int2(0, 0);
    }
    ph_headers(a, sm_box);
    grid.sync();
    GPL_STAMP(a, 1);
    // S1: grid parameters (every CTA derives the same values), cell counts, chunk-local scan of the bucket counts
    if (threadIdx.x == 0) {
        sm_g = grid_from_acc(a);
        if (blockIdx.x == 0) *a.gp = sm_g;
    }
    __syncthreads();
    ph_cells<0>(a, sm_g);
    grid_scan_local(a.nb, a.nb, a.P, a.partial, sm_scan);
    grid.sync();
    GPL_STAMP(a, 2);
    // S2: bucket bases (finishing the scan), bucket entry counts
    {
        const int64_t total = grid_scan_prefix(a.partial, sm_prefix, sm_scan);
        if (tid == 0) a.acc[ACC_BUCKETS] = (unsigned long long)total;
        __syncthreads();
        ph_buckets<0>(a, sm_prefix, ceil_div_dev(a.P > 0 ? a.P : 1, gridDim.x));
    }
    grid.sync();
    GPL_STAMP(a, 3);
    // S3: FP32 table plan
    ph_fast_plan(a);
    GPL_STAMP(a, 4);  // (one CTA's view: the kernel ends when the slowest CTA does)
}

__global__ void __launch_bounds__(kBuildThreads, 3) k_pip_build_fill(const BuildArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ int64_t sm_scan[kBuildThreads / 32 + 1];
    __shared__ int64_t sm_prefix[kMaxBuildCtas];
    __shared__ RasterSmem sm_raster;
    const GridParams g = *a.gp;
    const int64_t tid = (int64_t)blockIdx.x * kBuildThreads + threadIdx.x, nth = (int64_t)gridDim.x * kBuildThreads;
    const bool degenerate = g.inv_fw == 0.0 || g.inv_fh == 0.0;
    GPL_STAMP(a, 5);
    // T0: chunk-local scans (in place): cell counts -> cell starts, bucket counts -> bucket starts, FP32 slots ->
    // FP32 bases; raster cleared (all 3 on a degenerate grid: every point walks)
    grid_scan_local(a.cell_count, a.cell_count, a.n_cells, a.partial, sm_scan);
    grid_scan_local(a.bcount, a.bcount, a.n_buckets, a.partial + kMaxBuildCtas, sm_scan);
    grid_scan_local(a.fast_slots, a.fast_slots, a.P, a.partial + 2 * kMaxBuildCtas, sm_scan);
    {
        const int64_t n_words = (int64_t)g.fgy * g.wpr;
        const uint32_t fillv = degenerate ? 0xffffffffu : 0u;
        for (int64_t i = tid; i < n_words; i += nth) a.raster[i] = make_uint2(fillv, 0xffffffffu);  // y: set by ph_cell_finish
    }
    grid.sync();
    GPL_STAMP(a, 6);
    // T1: add the prefixes of the chunk totals; cursors for the fill passes
    {
        int64_t total = grid_scan_prefix(a.partial, sm_prefix, sm_scan);
        int64_t L = ceil_div_dev(a.n_cells > 0 ? a.n_cells : 1, gridDim.x);
        for (int64_t i = tid; i < a.n_cells; i += nth) {
            const int32_t v = a.cell_count[i] + (int32_t)sm_prefix[i / L];
            a.cell_count[i] = v, a.cell_cursor[i] = v;
        }
        if (tid == 0) a.cell_count[a.n_cells] = (int32_t)total;
        __syncthreads();
        total = grid_scan_prefix(a.partial + kMaxBuildCtas, sm_prefix, sm_scan);
        L = ceil_div_dev(a.n_buckets > 0 ? a.n_buckets : 1, gridDim.x);
        for (int64_t i = tid; i < a.n_buckets; i += nth) {
            const int32_t v = a.bcount[i] + (int32_t)sm_prefix[i / L];
            a.bcount[i] = v, a.bcursor[i] = v;
        }
        if (tid == 0) a.bcount[a.n_buckets] = (int32_t)total;
        __syncthreads();
        total = grid_scan_prefix(a.partial + 2 * kMaxBuildCtas, sm_prefix, sm_scan);
        L = ceil_div_dev(a.P > 0 ? a.P : 1, gridDim.x);
        for (int64_t i = tid; i < a.P; i += nth) a.fast_slots[i] += (int32_t)sm_prefix[i / L];
        __syncthreads();
    }
    grid.sync();
    GPL_STAMP(a, 7);
    const int32_t *cell_start = a.cell_count, *bstart = a.bcount;
    // T2: candidate lists of the cells, edge ids of the buckets (atomic cursors; sorted next)
    ph_cells<1>(a, g);
    ph_buckets<1>(a, nullptr, 1);
    grid.sync();
    GPL_STAMP(a, 8);
    // T3: candidate lists in ascending order; every y-bucket finished by one thread (sort, f64 records, FP32 lists)
    ph_sort_segments<int32_t>(a.items, cell_start, a.n_cells);
    ph_bucket_finish(a, bstart);
    ph_part_recs(a);
    for (int64_t b = tid; b < a.n_buckets; b += nth) a.bucket_range[b] = make_int2(bstart[b], bstart[b + 1]);
    grid.sync();
    GPL_STAMP(a, 9);
    // T4: cell records (need the sorted lists), raster
    ph_cell_finish(a, cell_start);
    GPL_STAMP(a, 10);
    ph_raster(a, g, cell_start, sm_raster);
    grid.sync();
    GPL_STAMP(a, 11);
    // T5: candidate #0 rows beside the raster codes (needs every cell record)
    ph_raster_cand(a, g);
}

// ------------------------------------------------------------------------------------------------
// the query kernels
// ------------------------------------------------------------------------------------------------
struct IndexView {
    const CellRec *cells;
    const int32_t *cell_items;
    const PartRec *parts;
    const int2 *bucket_range;
    const EdgeRec *entries;
    const int32_t *entry_ring;
    const float4 *fast;
    const uint2 *raster;
    const int2 *cand01;
    int32_t multi;  // polygon side is MULTIPOLYGON: several parts may share a row
    GridParams grid;
};
__device__ __forceinline__ int64_t coarse_cell(const GridParams &g, double px, double py) {
    const int32_t cx = fine_index(px, g.x0, g.inv_fw, g.fgx) >> g.rs, cy = fine_index(py, g.y0, g.inv_fh, g.fgy) >> g.rs;
    return (int64_t)cy * g.gx + cx;
}

// 256-bit loads (sm_100: LDG.E.256): one instruction, one L1 wavefront per distinct line
__device__ __forceinline__ void ld256(const void *p, double &a, double &b, double &c, double &d) {
    asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void ld256(const void *p, int32_t (&r)[8]) {
    asm("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
}

// One edge of geo's coord_pos_relative_to_ring loop, evaluated WITHOUT control flow: the orientation
// determinant and its static filter (Shewchuk stage A) are computed for every listed edge (nine FP64
// arithmetic ops, six compares) and the up/down rules are predicate arithmetic.  Whenever the filter
// cannot certify a NON-ZERO sign on an edge that actually straddles p.y — which includes every
// collinear (possible boundary) configuration — `undecided` is raised and the point is re-evaluated
// with the exact adaptive predicate and geo's boundary rule (k_pip_deferred / bucket_contains_exact).
// Probability ~1e-9 per edge on random data, so the hot loop has no branch, no call, no
// adaptive-precision code.  The winding contribution is identical to geo's for every decided edge.
__device__ __forceinline__ void edge_rule_fast(double sx, double sy, double ex, double ey, double px, double py, int &wn,
                                               bool &undecided) {
    const double dl = (sx - px) * (ey - py);
    const double dr = (sy - py) * (ex - px);
    const double det = dl - dr;
    // three ordinate comparisons decide everything geo's nested ifs decide:
    //   a = start.y <= p.y, b = end.y <= p.y, c = end.y >= p.y
    //   upward rule acts   <=> a && c ; counts <=> a && !b (end.y > p.y) && det > 0
    //   downward rule acts <=> !a && b ; counts <=> det < 0
    const bool a = sy <= py, b = ey <= py, c = ey >= py;
    const bool act = a ? c : b;
    const bool certain = fabs(det) > kCcwA * (fabs(dl) + fabs(dr));  // strict: det == 0 is never "certain"
    undecided = undecided || (act && !certain);
    wn += (int)(a && !b && det > 0.0) - (int)(!a && b && det < 0.0);
}

constexpr int kQueryThreads = 256;
constexpr int32_t kDeferred = -2;  // first_id marker: "the fast filter could not decide, see k_pip_deferred"

__device__ __forceinline__ void unpack_lite(const int32_t *r, PartLite &l) {
    l.xminf = __int_as_float(r[0]), l.xmaxf = __int_as_float(r[1]);
    l.yminf = __int_as_float(r[2]), l.inv_hf = __int_as_float(r[3]);
    l.nb_flags = r[4], l.bucket_base = r[5];
}
// x-range + y-bucket of one candidate part: false when no listed edge can act on p
__device__ __forceinline__ bool candidate_range(const IndexView &ix, const PartLite &l, double px, double py, int32_t &e0,
                                                int32_t &e1) {
    const int32_t nb = l.nb_flags & 0x00ffffff;
    const double t = (py - (double)l.yminf) * (double)l.inv_hf;
    // x outside the (outward rounded) range, or t < 0 (p.y < yminf <= ymin), or t >= nb + 1 (p.y > ymax)
    if (!(px >= (double)l.xminf && px <= (double)l.xmaxf) || t < 0.0 || !(t < (double)(nb + 1))) return false;
    const int32_t b = min((int32_t)t, nb - 1);
    const int2 range = __ldg(ix.bucket_range + l.bucket_base + b);
    e0 = range.x, e1 = range.y;
    return true;
}

// Serial walk of one bucket with the branch-free rule.  The loads of a batch of four edge records are
// issued back to back BEFORE any of them is consumed (four 256-bit loads in flight per lane): the first
// version let the compiler interleave load and use and paid one L2 round trip per edge.
// Returns Polygon::contains for this part when `undecided` stays false.
// HOLES: entries are grouped by ring (ascending ring index, 0 = exterior): exterior must wind, every
// hole must not.
template <bool HOLES>
__device__ __forceinline__ bool bucket_walk(const IndexView &ix, int32_t e0, int32_t e1, double px, double py, bool &undecided) {
    int wn = 0;
    bool und = false, ok = true;
    int32_t cur = 0;
    if (HOLES) {
        if (e0 == e1) return false;
        cur = __ldg(ix.entry_ring + e0);
        if (cur != 0) return false;  // no exterior edge near p.y: winding 0 => Outside
    }
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    for (int32_t k = e0; k < e1; k += 4) {
        double r[4][4];
        int32_t ring[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            // padding record: start.y = +inf, end.y = +inf never satisfies a or b => acts on nothing
            r[j][0] = r[j][1] = r[j][2] = r[j][3] = inf;
            ring[j] = cur;
            if (k + j < e1) {
                ld256(ix.entries + k + j, r[j][0], r[j][1], r[j][2], r[j][3]);
                if (HOLES) ring[j] = __ldg(ix.entry_ring + k + j);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (HOLES) {
                if (ring[j] != cur) {
                    ok = ok && (cur == 0 ? (wn != 0) : (wn == 0));
                    cur = ring[j];
                    wn = 0;
                }
            }
            edge_rule_fast(r[j][0], r[j][1], r[j][2], r[j][3], px, py, wn, und);
        }
    }
    undecided = undecided || und;
    if (HOLES) return ok && (cur == 0 ? (wn != 0) : (wn == 0));
    return wn != 0;
}

// ---- FP32 filter walk over the fixed-stride fast table ----------------------------------------------
// All quantities are relative to the part origin O = (xminf, yminf).  R bounds every |coordinate - O| that
// can occur on this path (edges lie in the bbox, p passed the x-range test and t < nb + 1 puts p.y at most
// one bucket above ymax: factor 2, absorbed below).  Each float difference u,v,w,z carries two conversions
// and one subtraction, each <= 2^-24 relative: |u - U| <= 3 * 2^-24 * 2R < eta := 2^-20 R.
//   ordinates  : |w| > eta and |v| > eta  =>  sign(w), sign(v) are the exact signs of (sy-py), (ey-py): the
//                predicates a, b, c of edge_rule_fast are known exactly and sy != py, ey != py;
//   determinant: |det - D| <= eta(|u|+|v|+|w|+|z| + 2 eta) + 2^-22(|uv|+|wz|)  (input perturbation plus
//                three float roundings) <= eta * 8.5 R + 2^-19 R^2 =: B  because |u|,|v|,|w|,|z| <= 2R;
//                so |det| > B  =>  sign(det) = sign(D) != 0.  B is one constant per (point, part).
// The relative-error model of the three float roundings needs normal numbers: the build only gives FP32 lists to
// parts with 2^-50 <= R <= 2^50 (ph_fast_plan), so eta >= 2^-70, B >= 2^-117 and any product below the normal range
// is far below B (never certified).
// Anything else raises `undecided`; the point is then recomputed from the f64 records with the exact
// predicate.  A definite answer is therefore always geo's answer.
__device__ __forceinline__ void fast_edge_rule(float4 e, float qx, float qy, float eta, float B, int &wn, bool &undecided) {
    const float u = e.x - qx, w = e.y - qy, z = e.z - qx, v = e.w - qy;
    const bool cert_y = fabsf(w) > eta && fabsf(v) > eta;
    const bool wl = w < 0.0f, vl = v < 0.0f;
    const bool act = wl != vl;
    const float det = u * v - w * z;
    undecided = undecided || !cert_y || (act && !(fabsf(det) > B));
    wn += (int)(act && wl && det > 0.0f) - (int)(act && !wl && det < 0.0f);
}
__device__ __forceinline__ void ld256f(const float4 *p, float4 &a, float4 &b) {
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
        : "l"(p));
}
// returns Polygon::contains for a plain part when `undecided` stays false
__device__ __forceinline__ bool fast_walk(const float4 *__restrict__ fast, const PartLite &l, double px, double py, bool &undecided) {
    const double xlo = (double)l.xminf, xhi = (double)l.xmaxf;
    if (!(px >= xlo && px <= xhi)) return false;
    const int32_t nb = l.nb_flags & 0x00ffffff;
    const bool right = px >= 0.5 * (xlo + xhi);  // which side's list (ph_fast_fill uses the same midpoint)
    // the bucket comes from the SAME double expression the build used (mono_index / candidate_range): a float
    // product could land one bucket off near a boundary and silently drop an edge whose end lies in the gap
    const double yrel = py - (double)l.yminf;
    const double t = yrel * (double)l.inv_hf;
    // t < 0 <=> p.y < yminf <= ymin ; t >= nb + 1 => p.y > ymax : no listed edge can act
    if (t < 0.0 || !(t < (double)(nb + 1))) return false;
    const int32_t b = min((int32_t)t, nb - 1);
    const float qx = __double2float_rn(right ? px - xlo : xhi - px), qy = __double2float_rn(yrel);
    const float4 *part = fast + (int64_t)l.bucket_base;
    const float4 *rec = part + (b * 2 + (right ? 0 : 1)) * kFastListRecs;
    const float R = fast_extent(l.xminf, l.xmaxf, l.inv_hf, nb);
    const float eta = 9.5367431640625e-07f * R;                          // 2^-20 R
    const float B = 1.01f * (8.5f * eta * R + 1.9073486328125e-06f * R * R);  // eta*8.5R + 2^-19 R^2
    const float inf = __int_as_float(0x7f800000);
    int wn = 0;
    bool und = !(B >= 1.17549435e-38f);  // defensive: the build never lists a part whose bounds leave the normal range
    // the list: header + (kFastListRecs - 1) edges, issued together; sentinels make the count irrelevant here
    float4 r[kFastListRecs];
#pragma unroll
    for (int j = 0; j < kFastListRecs / 2; ++j) ld256f(rec + 2 * j, r[2 * j], r[2 * j + 1]);
    const int32_t count = __float_as_int(r[0].x);
    const float4 *more = part + __float_as_int(r[0].y) - kFastListRecs;  // records kFastListRecs.. : the part's overflow area
#pragma unroll
    for (int j = 1; j < kFastListRecs; ++j) fast_edge_rule(r[j], qx, qy, eta, B, wn, und);
    for (int32_t k = kFastListRecs; k <= count; k += 4) {  // longer lists: four more edges per round (2 sectors)
        float4 t4[4];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            t4[2 * j] = make_float4(0.0f, inf, 0.0f, inf);
            t4[2 * j + 1] = t4[2 * j];
            if (k + 2 * j <= count) ld256f(more + k + 2 * j, t4[2 * j], t4[2 * j + 1]);  // slots past `count` are sentinels
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) fast_edge_rule(t4[j], qx, qy, eta, B, wn, und);
    }
    undecided = undecided || und;
    return wn != 0;
}

// The walk of ONE point that lies inside the union bbox: coarse cell -> candidates -> edge lists.
// MODE 0 (k_pip_stream): first (lowest containing row or -1) and cnt (all containing rows when want_count, else the walk
//         stops at the first hit); `undecided` = a filter could not certify something: the caller defers the point to
//         the exact kernel.
// MODE 1 (k_pip_pairs): write every (point, polygon) pair at lhs/rhs[w...]; undecided candidates are resolved in place
//         with the exact predicate (this mode is not the throughput path).
// LEAN (MODE 0 only): every part of the index is a plain POLYGON with FP32 lists (the host checks it), so the
// f64 bucket walk is compiled out and every candidate runs the FP32 walk.  A candidate that would still need the
// f64 walk is deferred (cannot happen when the host check holds; kept so that the kernel is correct on any index).
template <int MODE, bool LEAN>
__device__ __forceinline__ void walk_point(const IndexView &ix, const double2 p, const bool want_count, int32_t &first, int32_t &cnt,
                                           bool &undecided, uint64_t gi, int64_t w, uint64_t *__restrict__ lhs,
                                           uint64_t *__restrict__ rhs) {
    int32_t r[8];
    ld256(ix.cells + coarse_cell(ix.grid, p.x, p.y), r);
    const int32_t n_cand = r[0], first_part = r[1];
    int32_t last_geom = -1;
    for (int32_t c = 0; c < n_cand; ++c) {
        int32_t part = first_part, geom;
        PartLite lite;
        if (c == 0 && !ix.multi) {
            unpack_lite(r + 2, lite);
            if (lite.nb_flags & kFastBit) {  // single plain candidate: FP32 filter over the fast table
                bool und = false;
                bool inside = fast_walk(ix.fast, lite, p.x, p.y, und);
                if (und) {
                    if (MODE == 0) {
                        undecided = true;
                        return;
                    }
                    // pair mode: resolve in place from the f64 records
                    int32_t q[8];
                    ld256(ix.parts + first_part, q);
                    PartLite gl;
                    unpack_lite(q, gl);
                    int32_t a0, a1;
                    inside = candidate_range(ix, gl, p.x, p.y, a0, a1) &&
                             bucket_contains_exact(ix.entries, ix.entry_ring, false, a0, a1, p.x, p.y);
                }
                if (inside) {
                    if (MODE == 1) {
                        lhs[w] = gi;
                        rhs[w] = (uint64_t)first_part;
                        ++w;
                    } else {
                        first = first_part;
                        cnt = 1;
                    }
                }
                return;
            }
            if (LEAN && n_cand == 1) {  // a lone candidate without FP32 lists
                undecided = true;
                return;
            }
        }
        if (LEAN) {  // every candidate through its FP32 lists; anything else goes to the exact kernel
            int32_t q[8];
            const int32_t cand = __ldg(ix.cell_items + first_part + c);
            ld256(ix.parts + cand, q);
            PartLite fl;
            unpack_lite(q, fl);
            fl.bucket_base = q[7];  // PartRec::pad = base of the part's FP32 lists
            bool und = !(fl.nb_flags & kFastBit);
            const bool inside = !und && fast_walk(ix.fast, fl, p.x, p.y, und);
            if (und) {
                undecided = true;
                return;
            }
            if (inside) {
                if (first < 0) first = cand;
                ++cnt;
                if (!want_count) return;
            }
            continue;
        }
        if (c == 0 && !ix.multi) {
            if (n_cand > 1) part = __ldg(ix.cell_items + first_part);
            geom = part;
        } else {
            if (n_cand > 1) part = __ldg(ix.cell_items + first_part + c);
            int32_t q[8];
            ld256(ix.parts + part, q);
            unpack_lite(q, lite);
            geom = q[6];
        }
        if (geom == last_geom) continue;  // MultiPolygon::contains = any part; count rows once
        int32_t e0, e1;
        if (!candidate_range(ix, lite, p.x, p.y, e0, e1)) continue;
        bool und = false;
        bool inside = lite.nb_flags < 0 ? bucket_walk<true>(ix, e0, e1, p.x, p.y, und) : bucket_walk<false>(ix, e0, e1, p.x, p.y, und);
        if (und) {
            if (MODE == 0) {
                undecided = true;
                return;
            }
            inside = bucket_contains_exact(ix.entries, ix.entry_ring, lite.nb_flags < 0, e0, e1, p.x, p.y);
        }
        if (!inside) continue;
        last_geom = geom;
        if (MODE == 1) {
            lhs[w] = gi;
            rhs[w] = (uint64_t)geom;
            ++w;
        } else {
            if (first < 0) first = geom;
            ++cnt;
            if (!want_count) return;  // only the first hit is wanted
        }
    }
}

// Pair lists: the (point, polygon) pairs of point i go to lhs/rhs[pair_off[i]...] (the offsets are the exclusive scan of
// the per-point counts of a k_pip_stream pass).  One thread per point, every point walks (round 1's query kernel, MODE 1
// of walk_point).  32 consecutive points per warp (coalesced 512-byte read, software-prefetched one grid stride ahead).
constexpr int kPairsMinBlocks = 3;
__global__ void __launch_bounds__(kQueryThreads, kPairsMinBlocks) k_pip_pairs(const IndexView ix, const double2 *__restrict__ pts,
                                                                               const uint8_t *__restrict__ pts_validity, int64_t n_pts,
                                                                               const int64_t *__restrict__ pair_off,
                                                                               uint64_t *__restrict__ lhs, uint64_t *__restrict__ rhs) {
    const GridParams &g = ix.grid;
    const int64_t stride = (int64_t)gridDim.x * kQueryThreads;
    int64_t i = (int64_t)blockIdx.x * kQueryThreads + threadIdx.x;
    double2 p_next = make_double2(0.0, 0.0);
    if (i < n_pts) p_next = __ldcs(pts + i);  // read-once stream
    for (; i < n_pts; i += stride) {
        const double2 p = p_next;
        if (i + stride < n_pts) p_next = __ldcs(pts + i + stride);
        bool ok = p.x >= g.x0 && p.x <= g.x1 && p.y >= g.y0 && p.y <= g.y1;  // false for NaN (empty point)
        if (ok && pts_validity) ok = bit_get(pts_validity, i);
        int32_t first = -1, cnt = 0;
        bool undecided = false;
        if (ok) walk_point<1, false>(ix, p, false, first, cnt, undecided, (uint64_t)i, pair_off[i], lhs, rhs);
    }
}

// ---- the streaming kernel (MODE 0 of round 2) --------------------------------------------------------------
// Persistent warps; a warp takes tiles of 128 consecutive points (2 KB, two 256-bit loads per lane, the next tile
// prefetched into registers).  Per point: closed bbox test, fine cell by arithmetic, ONE 64-bit load of the raster
// word (four independent loads in flight per lane), then
//   code 0      -> -1
//   code 1      -> the row of the coarse cell's candidate #0: the word's upper half
//   code 2      -> the row of candidate #1 (one 8-byte load from the 80 KB cand01 table)
//   code 3      -> appended to the warp's shared-memory queue (ballot + popc compaction).
// Whenever the queue holds 32 points the warp walks them (walk_point) with all lanes active and overwrites their ids;
// the rest is drained at the end.  ids are written as 64-bit stores (two consecutive points per lane).
constexpr int kTilePts = 128;
constexpr int kQueueCap = kTilePts + 32;
constexpr int kStreamWarps = kQueryThreads / 32;
struct __align__(16) StreamSmem {
    double2 q_pts[kStreamWarps][kQueueCap];
    uint32_t q_idx[kStreamWarps][kQueueCap];
};
constexpr int kStreamMinBlocks = 3;
// The point stream and the raster gather (20 MB of random 8-byte words: no reuse an L1 could catch) are loaded without an
// L1 line, which leaves the L1 to the cell / part / edge records of the walk.  Query ms, config 2 / config 4: plain loads
// 0.846 / 0.856; raster gather L1::no_allocate 0.821 / 0.832; both 0.819 / 0.827; both plus an L2 evict-first policy on the
// stream 0.812 / 0.955.
__device__ __forceinline__ void ld256s_na(const double2 *p, double2 &a, double2 &b) {
    asm volatile("ld.global.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a.x), "=d"(a.y), "=d"(b.x), "=d"(b.y) : "l"(p));
}
__device__ __forceinline__ uint2 ldg_na(const uint2 *p) {
    uint2 v;
    asm("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    return v;
}
template <bool LEAN>
__global__ void __launch_bounds__(kQueryThreads, kStreamMinBlocks) k_pip_stream(const IndexView ix, const double2 *__restrict__ pts,
                                                                               const uint8_t *__restrict__ pts_validity, int64_t n_pts,
                                                                               int32_t *__restrict__ first_id, int32_t *__restrict__ count,
                                                                               unsigned long long *__restrict__ n_deferred,
                                                                               uint32_t *__restrict__ deferred_list, uint32_t list_cap,
                                                                               int vec_ok) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    StreamSmem &sm = *reinterpret_cast<StreamSmem *>(smem_raw);
    const GridParams &g = ix.grid;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double2 *q_pts = sm.q_pts[wid];
    uint32_t *q_idx = sm.q_idx[wid];
    int qn = 0;  // points waiting in this warp's queue (warp-uniform)
    const int64_t n_tiles = (n_pts + kTilePts - 1) / kTilePts;
    const int64_t n_warps = (int64_t)gridDim.x * kStreamWarps;
    int64_t tile = (int64_t)blockIdx.x * kStreamWarps + wid;
    const bool want_count = count != nullptr;

    auto walk_queued = [&](int e, bool active) {
        double2 p = make_double2(0.0, 0.0);
        uint32_t idx = 0;
        if (active) p = q_pts[e], idx = q_idx[e];
        __syncwarp();  // every lane holds its entry before the queue is written again
        if (active) {
            int32_t first = -1, cnt = 0;
            bool undecided = false;
            walk_point<0, LEAN>(ix, p, want_count, first, cnt, undecided, 0, 0, nullptr, nullptr);
            if (undecided) {
                first = kDeferred;
                const unsigned long long slot = atomicAdd(n_deferred, 1ULL);
                if (slot < list_cap) deferred_list[slot] = idx;  // chunk-relative index (chunks are < 2^32 points)
            }
            first_id[idx] = first;
            if (want_count) count[idx] = cnt;
        }
    };

    // k-th point of a lane inside a tile: pairs of consecutive points, two groups of 64
    auto slot_of = [&](int k) { return 2 * lane + (k & 1) + (k >> 1) * 64; };
    double2 nxt[4];
    auto load_tile = [&](int64_t t, double2 (&dst)[4]) {
        const int64_t base = t * kTilePts;
        if (vec_ok && base + kTilePts <= n_pts) {
            ld256s_na(pts + base + 2 * lane, dst[0], dst[1]);
            ld256s_na(pts + base + 64 + 2 * lane, dst[2], dst[3]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int64_t i = base + slot_of(k);
                dst[k] = i < n_pts ? __ldcs(pts + i) : make_double2(0.0, 0.0);
            }
        }
    };
    if (tile < n_tiles) load_tile(tile, nxt);
    for (; tile < n_tiles; tile += n_warps) {
        double2 p[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) p[k] = nxt[k];
        if (tile + n_warps < n_tiles) load_tile(tile + n_warps, nxt);
        const int64_t base = tile * kTilePts;
        // stage 1: fine cells and raster words
        int32_t fx[4], fy[4];
        uint2 word[4];
        bool ok[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int64_t i = base + slot_of(k);
            ok[k] = p[k].x >= g.x0 && p[k].x <= g.x1 && p[k].y >= g.y0 && p[k].y <= g.y1;  // false for NaN (empty point)
            if (i >= n_pts) ok[k] = false;
            if (ok[k] && pts_validity) ok[k] = bit_get(pts_validity, i);
            fx[k] = fine_index(p[k].x, g.x0, g.inv_fw, g.fgx), fy[k] = fine_index(p[k].y, g.y0, g.inv_fh, g.fgy);
            const uint2 *wp = ix.raster + (int64_t)fy[k] * g.wpr + (fx[k] >> 4);
            word[k] = ok[k] ? ldg_na(wp) : make_uint2(0u, 0u);
        }
        // stage 2: codes -> ids
        int32_t id[4];
        uint32_t code[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            code[k] = (word[k].x >> ((fx[k] & 15) * 2)) & 3u;
            id[k] = -1;
            if (code[k] == 1u || code[k] == 2u) {
                const int64_t cc = (int64_t)(fy[k] >> g.rs) * g.gx + (fx[k] >> g.rs);
                if (code[k] == 1u && word[k].y != 0xfffffffeu) {
                    id[k] = (int32_t)word[k].y;  // the candidate's row travels with the codes: no second gather
                } else {
                    // (staging the whole table in shared memory measured slower on config 2: 0.98 vs 0.90 ms)
                    const int2 cand = __ldg(ix.cand01 + cc);
                    id[k] = code[k] == 1u ? cand.x : cand.y;
                }
            }
        }
        // stage 3: ids out (the queued ones are overwritten by the walk)
        if (vec_ok && base + kTilePts <= n_pts) {
            __stcs(reinterpret_cast<int2 *>(first_id + base) + lane, make_int2(id[0], id[1]));
            __stcs(reinterpret_cast<int2 *>(first_id + base + 64) + lane, make_int2(id[2], id[3]));
            if (want_count) {
                __stcs(reinterpret_cast<int2 *>(count + base) + lane, make_int2(id[0] >= 0, id[1] >= 0));
                __stcs(reinterpret_cast<int2 *>(count + base + 64) + lane, make_int2(id[2] >= 0, id[3] >= 0));
            }
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int64_t i = base + slot_of(k);
                if (i < n_pts) {
                    first_id[i] = id[k];
                    if (want_count) count[i] = id[k] >= 0;
                }
            }
        }
        // stage 4: queue the walkers
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool q = code[k] == 3u;
            const unsigned m = __ballot_sync(0xffffffffu, q);
            if (q) {
                const int pos = qn + __popc(m & ((1u << lane) - 1u));
                q_pts[pos] = p[k];
                q_idx[pos] = (uint32_t)(base + slot_of(k));
            }
            qn += __popc(m);
        }
        __syncwarp();
        while (qn >= 32) {
            qn -= 32;
            walk_queued(qn + lane, true);
        }
    }
    if (qn > 0) walk_queued(lane, lane < qn);
}

// Exact re-evaluation of the points the walk marked kDeferred (those whose filters could not
// certify an ordinate relation or an orientation that mattered: points within ~1e-6 of an edge or of a
// vertex ordinate, relative to the part size).  Launched after every query; exits at once when the
// counter is zero.  One thread per deferred point, taken from the list the query kernel appended to; if
// the list overflowed, the id column is scanned for the marker instead.
__device__ __forceinline__ void deferred_point(const IndexView &ix, const double2 *__restrict__ pts, int64_t i,
                                               int32_t *__restrict__ first_id, int32_t *__restrict__ count) {
    const double2 p = pts[i];
    const CellRec cell = ix.cells[coarse_cell(ix.grid, p.x, p.y)];
    int32_t first = -1, cnt = 0, last_geom = -1;
    for (int32_t c = 0; c < cell.count; ++c) {
        const int32_t part = cell.count == 1 ? cell.first : ix.cell_items[cell.first + c];
        const PartRec rec = ix.parts[part];
        if (rec.geom == last_geom) continue;
        int32_t e0, e1;
        if (!candidate_range(ix, rec.lite, p.x, p.y, e0, e1)) continue;
        if (!bucket_contains_exact(ix.entries, ix.entry_ring, rec.lite.nb_flags < 0, e0, e1, p.x, p.y)) continue;
        last_geom = rec.geom;
        if (first < 0) first = rec.geom;
        ++cnt;
        if (count == nullptr) break;
    }
    first_id[i] = first;
    if (count) count[i] = cnt;
}
__global__ void __launch_bounds__(256) k_pip_deferred(const IndexView ix, const double2 *__restrict__ pts, int64_t n_pts,
                                                      int32_t *__restrict__ first_id, int32_t *__restrict__ count,
                                                      unsigned long long *__restrict__ n_deferred,
                                                      const uint32_t *__restrict__ deferred_list, uint32_t list_cap,
                                                      unsigned long long *__restrict__ n_deferred_total) {
    const unsigned long long nd = *n_deferred;
    if (nd == 0ULL) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (nd <= list_cap) {
        for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < (int64_t)nd; k += stride)
            deferred_point(ix, pts, (int64_t)deferred_list[k], first_id, count);
    } else {
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pts; i += stride)
            if (first_id[i] == kDeferred) deferred_point(ix, pts, i, first_id, count);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_deferred_total) atomicAdd(n_deferred_total, nd);
}

// per-polygon hit counts (config 4's all-reduce input).  Counts are privatised per CTA in shared memory
// (32-bit, up to kHistSmemBins bins) and flushed once: 36 M global atomics on 10 k addresses become 1184 x 10 k.
constexpr int kHistSmemBins = 48 * 1024;
__global__ void __launch_bounds__(512) k_histogram(const int32_t *__restrict__ ids, int64_t n, unsigned long long *__restrict__ counts,
                                                   int64_t n_polys, int use_smem) {
    extern __shared__ unsigned int s_bins[];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (use_smem) {
        for (int64_t b = threadIdx.x; b < n_polys; b += blockDim.x) s_bins[b] = 0u;
        __syncthreads();
    }
    auto add = [&](int32_t id) {
        if (id >= 0 && id < n_polys) {
            if (use_smem) atomicAdd(&s_bins[id], 1u);
            else atomicAdd(&counts[id], 1ULL);
        }
    };
    // four ids per thread and iteration (one 128-bit load; cudaMalloc'd columns are 16-byte aligned)
    const int64_t n4 = ((reinterpret_cast<uintptr_t>(ids) & 15) == 0) ? n / 4 : 0;
    const int4 *ids4 = reinterpret_cast<const int4 *>(ids);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += stride) {
        const int4 v = __ldcs(ids4 + i);
        add(v.x), add(v.y), add(v.z), add(v.w);
    }
    for (int64_t i = n4 * 4 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) add(__ldcs(ids + i));
    if (use_smem) {
        __syncthreads();
        for (int64_t b = threadIdx.x; b < n_polys; b += blockDim.x) {
            const unsigned int v = s_bins[b];
            if (v) atomicAdd(&counts[b], (unsigned long long)v);
        }
    }
}

static IndexView view_of(const gpl_pip_index *idx) {
    IndexView v;
    v.cells = idx->cells, v.cell_items = idx->cell_overflow, v.parts = idx->parts;
    v.bucket_range = idx->bucket_range, v.entries = idx->entries, v.entry_ring = idx->entry_ring;
    v.fast = idx->fast;
    v.raster = idx->raster, v.cand01 = idx->cand01;
    v.multi = idx->multi ? 1 : 0;
    v.grid = idx->grid;
    return v;
}

// pair kernel: 148 SMs x 8 CTAs, grid-stride over the points
static int pairs_grid(int64_t n) {
    return (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n, kQueryThreads), (int64_t)kSMs * 8));
}
// streaming kernel: exactly the resident CTAs (persistent warps, one tile of 128 points per warp and iteration)
template <bool LEAN>
static void launch_stream(const IndexView &v, const double2 *pts, const uint8_t *val, int64_t m, int32_t *first, int32_t *cnt,
                          const gpl_pip_index *idx, int vec_ok, cudaStream_t stream) {
    constexpr size_t smem = sizeof(StreamSmem);
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_pip_stream<LEAN>, kQueryThreads, smem) != cudaSuccess || occ < 1) occ = 1;
    (void)cudaGetLastError();
    const int64_t want = ceil_div(ceil_div(m, kTilePts), kStreamWarps);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)kSMs * occ));
    k_pip_stream<LEAN><<<grid, kQueryThreads, smem, stream>>>(v, pts, val, m, first, cnt, idx->n_deferred, idx->deferred_list,
                                                              idx->deferred_cap, vec_ok);
}
// counts[id] += 1 for every id in [0, n_polys) of the column ids[0, n)
static int launch_histogram(gpl_ctx *ctx, const int32_t *ids, int64_t n, unsigned long long *counts, int64_t n_polys,
                            cudaStream_t stream) {
    const bool use_smem = n_polys <= kHistSmemBins;
    const size_t dyn = use_smem ? sizeof(unsigned int) * (size_t)n_polys : 0;
    if (dyn > 48 * 1024) GPL_CUDA(cudaFuncSetAttribute(k_histogram, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    const int per_sm = use_smem ? (int)std::max<size_t>(1, std::min<size_t>(4, (200 * 1024) / std::max<size_t>(dyn, 1))) : 4;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n, 2048), (int64_t)kSMs * per_sm));
    k_histogram<<<grid, 512, dyn, stream>>>(ids, n, counts, n_polys, use_smem ? 1 : 0);
    ctx->launches++;
    return GPL_OK;
}
// hist (optional, device, n_geoms u64): += number of points whose first containing row is that polygon.  The counts are a
// separate pass over the id column (k_histogram: 0.1 ms per 100 M ids): shared-memory bins fused into the streaming kernel
// measured slower on config 2 (+0.22 ms).
int pip_query(gpl_ctx *ctx, const gpl_pip_index *idx, const double *pts_dev, const uint8_t *validity_dev, int64_t n,
              int32_t *first_dev, int32_t *count_dev, cudaStream_t stream, unsigned long long *hist = nullptr) {
    if (n == 0) return GPL_OK;
    const double2 *pts = reinterpret_cast<const double2 *>(pts_dev);
    const IndexView v = view_of(idx);
    // the deferred list holds chunk-relative uint32 indices: process at most 2^31 points per launch pair
    const int64_t kMaxChunk = 1LL << 31;
    for (int64_t lo = 0; lo < n; lo += kMaxChunk) {
        const int64_t m = std::min(kMaxChunk, n - lo);
        const uint32_t cap = (uint32_t)std::min<int64_t>(std::max<int64_t>(m / 16, 1 << 16), 1 << 26);
        if (idx->deferred_cap < cap) {
            gpl_pip_index *mut = const_cast<gpl_pip_index *>(idx);
            ctx->release(mut->deferred_list);
            void *q = nullptr;
            GPL_TRY(ctx->alloc(sizeof(uint32_t) * (size_t)cap, &q));
            mut->deferred_list = (uint32_t *)q;
            mut->deferred_cap = cap;
        }
        GPL_CUDA(cudaMemsetAsync(idx->n_deferred, 0, sizeof(unsigned long long), stream));
        const uint8_t *val = validity_dev ? validity_dev + lo / 8 : nullptr;
        int32_t *cnt = count_dev ? count_dev + lo : nullptr;
        cudaEvent_t t0 = nullptr, t1 = nullptr;
        if (ctx->kt_on && ctx->kernel_timing_pair(&t0, &t1)) GPL_CUDA(cudaEventRecord(t0, stream));
        // 256-bit point loads and 64-bit id stores need 32- / 8-byte aligned columns (cudaMalloc'd ones are)
        const int vec_ok = ((reinterpret_cast<uintptr_t>(pts + lo) & 31) == 0 && (reinterpret_cast<uintptr_t>(first_dev + lo) & 7) == 0 &&
                            (cnt == nullptr || (reinterpret_cast<uintptr_t>(cnt) & 7) == 0))
                               ? 1
                               : 0;
        if (idx->lean_ok) launch_stream<true>(v, pts + lo, val, m, first_dev + lo, cnt, idx, vec_ok, stream);
        else launch_stream<false>(v, pts + lo, val, m, first_dev + lo, cnt, idx, vec_ok, stream);
        if (t1) GPL_CUDA(cudaEventRecord(t1, stream));
        k_pip_deferred<<<kSMs * 8, 256, 0, stream>>>(v, pts + lo, m, first_dev + lo, cnt, idx->n_deferred, idx->deferred_list, idx->deferred_cap,
                                                     idx->n_deferred + 1);
        ctx->launches += 2;
        if (hist) GPL_TRY(launch_histogram(ctx, first_dev + lo, m, hist, idx->n_geoms, stream));
    }
    GPL_CUDA(cudaGetLastError());
    return GPL_OK;
}

}  // namespace gpl

using namespace gpl;

// Keep the hot part of the index slab resident in the 126 MB L2 while 1.6 GB of points stream past it: mark it
// as a persisting access-policy window on the context stream.  Best effort: failures only cost performance.  The
// device-wide carve-out only ever grows while the context lives and is restored by gpl_ctx_destroy; the window is
// dropped and the persisting lines are released when the index that set them is freed (neither call waits for running
// kernels: they are cache hints).
static void l2_pin(gpl_pip_index *idx, bool on) {
    gpl_ctx *ctx = idx->ctx;
    if (ctx->l2_persist_max == 0 || ctx->l2_window_max == 0) return;
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    if (on) {
        const size_t want = idx->hot_bytes ? idx->hot_bytes : idx->slab_bytes;
        size_t carve = std::min<size_t>(want, ctx->l2_persist_max);
        if (!ctx->l2_limit_saved) {
            size_t prev = 0;
            if (cudaDeviceGetLimit(&prev, cudaLimitPersistingL2CacheSize) == cudaSuccess) {
                ctx->l2_prev_limit = prev;
                ctx->l2_limit_saved = true;
                ctx->l2_cur_limit = prev;
            }
        }
        if (carve > ctx->l2_cur_limit) {
            (void)cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
            ctx->l2_cur_limit = carve;
        }
        carve = std::min(carve, ctx->l2_cur_limit);
        size_t win = std::min<size_t>(want, ctx->l2_window_max);
        attr.accessPolicyWindow.base_ptr = idx->slab;
        attr.accessPolicyWindow.num_bytes = win;
        attr.accessPolicyWindow.hitRatio = win > 0 ? std::min(1.0f, (float)carve / (float)win) : 0.0f;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        ctx->l2_pinned = idx->slab;
    } else {
        if (ctx->l2_pinned != idx->slab) return;  // another index owns the window now
        attr.accessPolicyWindow.num_bytes = 0;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
        ctx->l2_pinned = nullptr;
    }
    (void)cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &attr);
    if (!on) (void)cudaCtxResetPersistingL2Cache();
    (void)cudaGetLastError();
}

extern "C" void gpl_pip_index_free(gpl_pip_index *idx) {
    if (!idx) return;
    if (idx->slab) l2_pin(idx, false);
    idx->ctx->release(idx->slab);
    idx->ctx->release(idx->deferred_list);
    delete idx;
}
extern "C" int64_t gpl_pip_index_bytes(const gpl_pip_index *idx) { return idx ? idx->bytes : 0; }

// diagnostic counters: out[0] = points the exact kernel re-evaluated since the index was built (all queries),
// out[1] = fine cells per axis, out[2] = log2(fine cells per coarse cell and axis), out[3] = raster cells coded 3,
// out[4] = raster cells coded 1 or 2, out[5] = parts without FP32 lists, out[6] = index bytes, out[7] = coarse cells per axis.
// Synchronises the context stream.
namespace gpl {
__global__ void k_raster_stats(const uint2 *__restrict__ raster, int64_t n_words, unsigned long long *__restrict__ out) {
    unsigned long long walk = 0, inside = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t w = raster[i].x, lo = w & 0x55555555u, hi = (w >> 1) & 0x55555555u;
        walk += __popc(lo & hi);
        inside += __popc(lo ^ hi);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        walk += __shfl_down_sync(0xffffffffu, walk, o);
        inside += __shfl_down_sync(0xffffffffu, inside, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(out, walk);
        atomicAdd(out + 1, inside);
    }
}
}  // namespace gpl
extern "C" int gpl_pip_index_stats(gpl_ctx *ctx, const gpl_pip_index *idx, int64_t *out8) {
    GPL_REQUIRE(ctx && idx && out8, GPL_ERR_INVALID_ARG, "gpl_pip_index_stats: NULL argument");
    GPL_CUDA(cudaSetDevice(ctx->device));
    Scratch<unsigned long long> tmp;
    GPL_TRY(tmp.get(ctx, 2));
    GPL_CUDA(cudaMemsetAsync(tmp.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
    const int64_t n_words = (int64_t)idx->grid.fgy * idx->grid.wpr;
    if (n_words > 0) {
        k_raster_stats<<<kSMs * 4, 256, 0, ctx->stream>>>(idx->raster, n_words, tmp.p);
        ctx->launches++;
    }
    unsigned long long h[3] = {0, 0, 0};
    GPL_CUDA(cudaMemcpyAsync(h, tmp.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaMemcpyAsync(h + 2, idx->n_deferred + 1, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    out8[0] = (int64_t)h[2];
    out8[1] = idx->grid.fgx;
    out8[2] = idx->grid.rs;
    out8[3] = (int64_t)h[0];
    out8[4] = (int64_t)h[1];
    out8[5] = idx->n_not_fast;
    out8[6] = idx->bytes;
    out8[7] = idx->grid.gx;
    return GPL_OK;
}

// build timeline of the FILL kernel (diagnostics): out12[k] = microseconds from the kernel's start to phase boundary k
// (5 = start, 6..9 = after grid barriers T0..T3, 10 = cell records done, 11 = raster done); synchronises the stream.
extern "C" int gpl_pip_index_phases(gpl_ctx *ctx, const gpl_pip_index *idx, double *out12) {
    GPL_REQUIRE(ctx && idx && out12, GPL_ERR_INVALID_ARG, "gpl_pip_index_phases: NULL argument");
    GPL_CUDA(cudaSetDevice(ctx->device));
    unsigned long long h[16];
    GPL_CUDA(cudaMemcpyAsync(h, idx->phase_t, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 12; ++k) out12[k] = k >= 5 ? (double)(h[k] - h[5]) * 1e-3 : 0.0;
    return GPL_OK;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

template <typename K>
static int coop_grid(K kernel) {
    int occ = 0, dev = 0, sms = kSMs;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kBuildThreads, 0) != cudaSuccess || occ < 1) occ = 1;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) sms = kSMs;
    (void)cudaGetLastError();
    return std::min(kMaxBuildCtas, sms * std::min(occ, 4));  // every CTA must be resident: grid-wide barriers
}

extern "C" int gpl_pip_index_build(gpl_ctx *ctx, const gpl_array *polys, gpl_pip_index **out) {
    GPL_REQUIRE(ctx && polys && out, GPL_ERR_INVALID_ARG, "gpl_pip_index_build: NULL argument");
    GPL_REQUIRE(polys->type == GPL_POLYGON || polys->type == GPL_MULTIPOLYGON, GPL_ERR_INVALID_TYPE,
                "Expected Polygon or MultiPolygon (found geometry type %d)", polys->type);
    GPL_CUDA(cudaSetDevice(ctx->device));
    const int type = polys->type;
    const int64_t P = type == GPL_POLYGON ? polys->n_geoms : polys->n_parts;
    GPL_REQUIRE(P < (1LL << 31) && polys->n_coords < (1LL << 31), GPL_ERR_UNSUPPORTED,
                "polygon side of a broadcast join is limited to 2^31 parts/coords");
    gpl_pip_index *idx = new gpl_pip_index();
    idx->ctx = ctx, idx->polys = polys, idx->n_parts = P, idx->n_geoms = polys->n_geoms;
    auto fail = [&](int rc) {
        gpl_pip_index_free(idx);
        return rc;
    };
#define TRYF(expr)                         \
    do {                                   \
        int rc__ = (expr);                 \
        if (rc__ != GPL_OK) return fail(rc__); \
    } while (0)
#define CUDAF(expr)                                                                     \
    do {                                                                                \
        cudaError_t e__ = (expr);                                                       \
        if (e__ != cudaSuccess) return fail(cuda_fail(e__, #expr, __FILE__, __LINE__)); \
    } while (0)

    const int64_t Pa = P > 0 ? P : 1;
    cudaStream_t st = ctx->stream;
    static const int grid_count = coop_grid(k_pip_build_count), grid_fill = coop_grid(k_pip_build_fill);

    // coarse grid: about one cell per part.  Fine grid: 2^rs x 2^rs cells per coarse cell, as fine as a budget of
    // raster cells allows (8 bytes per 16 cells: 64 M cells = 32 MB, L2-resident next to the FP32 table), at most 2^7, and at
    // most 2^20 fine cells per axis (the error analysis of the raster assumes it).
    constexpr int kRasterLog2Max = 7;
    constexpr int64_t kRasterCells = 64LL << 20;
    int64_t G = (int64_t)ceil(sqrt((double)Pa));
    if (G < 1) G = 1;
    if (G > 2048) G = 2048;
    const int64_t n_cells = G * G;
    int rs = kRasterLog2Max;
    while (rs > 0 && (((G << rs) > (1 << 20)) || ((G << rs) * (G << rs) > kRasterCells))) --rs;

    // ---- phase 1 (scratch): bboxes, grid, cell counts, bucket counts, FP32 plan --------------------------------
    BuildArgs a;
    memset(&a, 0, sizeof(a));
    a.type = type, a.P = P, a.n_geoms = polys->n_geoms;
    a.xy = reinterpret_cast<const double2 *>(polys->xy);
    a.geom_off = polys->geom_off, a.part_off = polys->part_off, a.ring_off = polys->ring_off, a.validity = polys->validity;
    a.G = (int32_t)G, a.rs = rs, a.n_cells = n_cells;
    // sum of n_buckets <= P + n_coords * 100 / kSlotsX100 + 1 without a host round trip
    a.NB_cap = Pa + (polys->n_coords * 100) / kSlotsX100 + 1;
    Scratch<PartHeader> hdr;
    Scratch<GridParams> gp;
    Scratch<int32_t> nb, cell_count, cell_cursor, bcount, bcursor, fast_c, fast_slots;
    Scratch<int2> side_count, ovf_off;
    Scratch<int32_t> bucket_part;
    Scratch<int64_t> partial;
    Scratch<unsigned long long> acc;
    TRYF(hdr.get(ctx, (size_t)Pa));
    TRYF(gp.get(ctx, 1));
    TRYF(nb.get(ctx, (size_t)Pa + 1));
    TRYF(partial.get(ctx, (size_t)4 * kMaxBuildCtas));
    TRYF(cell_count.get(ctx, (size_t)n_cells + 1));
    TRYF(bcount.get(ctx, (size_t)a.NB_cap + 1));
    TRYF(side_count.get(ctx, (size_t)a.NB_cap + 1));
    TRYF(ovf_off.get(ctx, (size_t)a.NB_cap + 1));
    TRYF(bucket_part.get(ctx, (size_t)a.NB_cap + 1));
    TRYF(fast_c.get(ctx, (size_t)Pa + 1));
    TRYF(fast_slots.get(ctx, (size_t)Pa + 1));
    TRYF(acc.get(ctx, ACC_COUNT));
    a.hdr = hdr.p, a.gp = gp.p, a.nb = nb.p, a.partial = partial.p, a.cell_count = cell_count.p, a.bcount = bcount.p;
    a.side_count = side_count.p, a.fast_c = fast_c.p, a.fast_slots = fast_slots.p, a.acc = acc.p;
    a.ovf_off = ovf_off.p, a.bucket_part = bucket_part.p;
    CUDAF(cudaMemsetAsync(acc.p, 0, sizeof(unsigned long long) * ACC_COUNT, st));
    {
        void *args[] = {&a};
        CUDAF(cudaLaunchCooperativeKernel((void *)k_pip_build_count, dim3(grid_count), dim3(kBuildThreads), args, 0, st));
        ctx->launches++;
    }
    // the data-dependent sizes + the grid parameters: one small D2H (index build is once per join)
    unsigned long long h_acc[ACC_COUNT];
    CUDAF(cudaMemcpyAsync(h_acc, acc.p, sizeof(h_acc), cudaMemcpyDeviceToHost, st));
    CUDAF(cudaMemcpyAsync(&idx->grid, gp.p, sizeof(GridParams), cudaMemcpyDeviceToHost, st));
    CUDAF(cudaStreamSynchronize(st));
    idx->n_overflow = (int64_t)h_acc[ACC_ITEMS];  // all cell items
    idx->n_buckets = (int64_t)h_acc[ACC_BUCKETS];
    idx->n_entries = (int64_t)h_acc[ACC_ENTRIES];
    idx->n_fast = (int64_t)h_acc[ACC_FAST];
    if (idx->n_fast >= (1LL << 31) || idx->n_entries >= (1LL << 31) || idx->n_overflow >= (1LL << 31)) {
        set_error("join index too large (%lld edge records, %lld cell items)", (long long)idx->n_entries,
                  (long long)idx->n_overflow);
        return fail(GPL_ERR_UNSUPPORTED);
    }
    idx->any_holes = h_acc[ACC_HOLES] != 0;  // set on the device: ring counts alone cannot tell (an empty polygon next to one with a hole)
    idx->n_not_fast = (int64_t)h_acc[ACC_NOT_FAST];
    idx->multi = type == GPL_MULTIPOLYGON;

    // ---- phase 2: one slab, filled in place ----------------------------------------------------------
    size_t off = 0;
    auto carve = [&](size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    // hot structures first: the L2-persisting window covers [0, hot_bytes) only, so the f64 records that
    // just the exact kernel reads do not compete for the cache with the tables every point touches
    const size_t raster_words = (size_t)idx->grid.fgy * (size_t)idx->grid.wpr;
    const size_t o_raster = carve(sizeof(uint2) * (raster_words + 1));
    const size_t o_cand = carve(sizeof(int2) * n_cells);
    const size_t o_cells = carve(sizeof(CellRec) * n_cells);
    const size_t o_fast = carve(sizeof(float4) * (idx->n_fast + 8));
    const size_t o_parts = carve(sizeof(PartRec) * Pa);
    const size_t o_brange = carve(sizeof(int2) * (idx->n_buckets + 1));
    const size_t o_items = carve(sizeof(int32_t) * (idx->n_overflow + 1));
    const size_t o_defer = carve(2 * sizeof(unsigned long long));
    const size_t o_phase = carve(16 * sizeof(unsigned long long));
    const bool all_fast = idx->n_fast > 0 && !idx->multi && !idx->any_holes;
    // POLYGON rows without holes, every valid part has FP32 lists (cells may hold several candidates)
    idx->lean_ok = all_fast && idx->n_not_fast == 0;
    const size_t hot_mark = off;
    const size_t o_entries = carve(sizeof(EdgeRec) * (idx->n_entries + 1));
    const size_t o_ring = idx->any_holes ? carve(sizeof(int32_t) * (idx->n_entries + 1)) : 0;
    idx->hot_bytes = all_fast ? hot_mark : 0;  // 0: pin the whole slab (general-path parts read the f64 records)
    void *q = nullptr;
    TRYF(ctx->alloc(off, &q));
    idx->slab = (uint8_t *)q;
    idx->slab_bytes = off;
    idx->raster = (uint2 *)(idx->slab + o_raster);
    idx->cand01 = (int2 *)(idx->slab + o_cand);
    idx->cells = (CellRec *)(idx->slab + o_cells);
    idx->parts = (PartRec *)(idx->slab + o_parts);
    idx->bucket_range = (int2 *)(idx->slab + o_brange);
    idx->entries = (EdgeRec *)(idx->slab + o_entries);
    idx->cell_overflow = (int32_t *)(idx->slab + o_items);
    idx->entry_ring = idx->any_holes ? (int32_t *)(idx->slab + o_ring) : nullptr;
    idx->n_deferred = (unsigned long long *)(idx->slab + o_defer);
    idx->phase_t = (unsigned long long *)(idx->slab + o_phase);
    idx->fast = (float4 *)(idx->slab + o_fast);
    idx->bytes = (int64_t)off;

    Scratch<int64_t> entry_edge;
    TRYF(entry_edge.get(ctx, (size_t)idx->n_entries + 1));
    TRYF(cell_cursor.get(ctx, (size_t)n_cells + 1));
    TRYF(bcursor.get(ctx, (size_t)idx->n_buckets + 1));
    a.n_buckets = idx->n_buckets, a.n_entries = idx->n_entries;
    a.cell_cursor = cell_cursor.p, a.bcursor = bcursor.p, a.entry_edge = entry_edge.p;
    a.cells = idx->cells, a.cand01 = idx->cand01, a.items = idx->cell_overflow, a.parts = idx->parts;
    a.bucket_range = idx->bucket_range, a.entries = idx->entries, a.entry_ring = idx->entry_ring, a.fast = idx->fast;
    a.raster = idx->raster, a.n_deferred = idx->n_deferred, a.phase_t = idx->phase_t;
    CUDAF(cudaMemsetAsync(idx->n_deferred, 0, 2 * sizeof(unsigned long long), st));
    {
        void *args[] = {&a};
        CUDAF(cudaLaunchCooperativeKernel((void *)k_pip_build_fill, dim3(grid_fill), dim3(kBuildThreads), args, 0, st));
        ctx->launches++;
    }
    CUDAF(cudaGetLastError());
    // No final synchronize: the scratch buffers above return to the context cache, which only ever hands them
    // to work enqueued later on this same stream (stream-ordered reuse), and every consumer of the index
    // launches on this stream too.
    l2_pin(idx, true);
    *out = idx;
    return GPL_OK;
#undef TRYF
#undef CUDAF
}

extern "C" int gpl_contains_join(gpl_ctx *ctx, const gpl_pip_index *idx, const double *points_xy, int64_t n_points,
                                 int32_t *first_id, int32_t *count, int mem) {
    GPL_REQUIRE(ctx && idx && first_id && (points_xy || n_points == 0), GPL_ERR_INVALID_ARG, "gpl_contains_join: NULL argument");
    GPL_CUDA(cudaSetDevice(ctx->device));
    if (n_points == 0) return GPL_OK;
    if (mem == GPL_DEVICE) return pip_query(ctx, idx, points_xy, nullptr, n_points, first_id, count, ctx->stream);
    // host buffers: plain (unpipelined) path — copy in, run, copy out.  gpl_contains_join_host overlaps them.
    Scratch<double> pts;
    Scratch<int32_t> ids, cnt;
    GPL_TRY(pts.get(ctx, (size_t)n_points * 2));
    GPL_TRY(ids.get(ctx, (size_t)n_points));
    if (count) GPL_TRY(cnt.get(ctx, (size_t)n_points));
    GPL_CUDA(cudaMemcpyAsync(pts.p, points_xy, sizeof(double) * 2 * n_points, cudaMemcpyHostToDevice, ctx->stream));
    GPL_TRY(pip_query(ctx, idx, pts.p, nullptr, n_points, ids.p, count ? cnt.p : nullptr, ctx->stream));
    GPL_CUDA(cudaMemcpyAsync(first_id, ids.p, sizeof(int32_t) * n_points, cudaMemcpyDeviceToHost, ctx->stream));
    if (count) GPL_CUDA(cudaMemcpyAsync(count, cnt.p, sizeof(int32_t) * n_points, cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    return GPL_OK;
}

extern "C" int gpl_contains_join_counts(gpl_ctx *ctx, const gpl_pip_index *idx, const double *points_xy, int64_t n_points,
                                        int32_t *first_id, uint64_t *counts, int mem) {
    GPL_REQUIRE(ctx && idx && first_id && counts && (points_xy || n_points == 0), GPL_ERR_INVALID_ARG,
                "gpl_contains_join_counts: NULL argument");
    GPL_CUDA(cudaSetDevice(ctx->device));
    if (n_points == 0) return GPL_OK;
    if (mem == GPL_DEVICE)
        return pip_query(ctx, idx, points_xy, nullptr, n_points, first_id, nullptr, ctx->stream, reinterpret_cast<unsigned long long *>(counts));
    Scratch<double> pts;
    Scratch<int32_t> ids;
    Scratch<unsigned long long> cnt;
    const size_t ng = (size_t)idx->n_geoms;
    GPL_TRY(pts.get(ctx, (size_t)n_points * 2));
    GPL_TRY(ids.get(ctx, (size_t)n_points));
    GPL_TRY(cnt.get(ctx, ng));
    GPL_CUDA(cudaMemcpyAsync(pts.p, points_xy, sizeof(double) * 2 * n_points, cudaMemcpyHostToDevice, ctx->stream));
    GPL_CUDA(cudaMemcpyAsync(cnt.p, counts, sizeof(uint64_t) * ng, cudaMemcpyHostToDevice, ctx->stream));
    GPL_TRY(pip_query(ctx, idx, pts.p, nullptr, n_points, ids.p, nullptr, ctx->stream, cnt.p));
    GPL_CUDA(cudaMemcpyAsync(first_id, ids.p, sizeof(int32_t) * n_points, cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaMemcpyAsync(counts, cnt.p, sizeof(uint64_t) * ng, cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    return GPL_OK;
}

extern "C" int gpl_contains_join_array(gpl_ctx *ctx, const gpl_pip_index *idx, const gpl_array *points, int32_t *first_id,
                                       int32_t *count, int mem) {
    GPL_REQUIRE(ctx && idx && points && first_id, GPL_ERR_INVALID_ARG, "gpl_contains_join_array: NULL argument");
    GPL_REQUIRE(points->type == GPL_POINT, GPL_ERR_INVALID_TYPE, "Expected Point (found geometry type %d)", points->type);
    GPL_CUDA(cudaSetDevice(ctx->device));
    int64_t n = points->n_geoms;
    if (n == 0) return GPL_OK;
    if (mem == GPL_DEVICE) return pip_query(ctx, idx, points->xy, points->validity, n, first_id, count, ctx->stream);
    Scratch<int32_t> ids, cnt;
    GPL_TRY(ids.get(ctx, (size_t)n));
    if (count) GPL_TRY(cnt.get(ctx, (size_t)n));
    GPL_TRY(pip_query(ctx, idx, points->xy, points->validity, n, ids.p, count ? cnt.p : nullptr, ctx->stream));
    GPL_CUDA(cudaMemcpyAsync(first_id, ids.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (count) GPL_CUDA(cudaMemcpyAsync(count, cnt.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    return GPL_OK;
}

// The (point, polygon) pair list of the device points pts[0, n) (validity optional; n > 0): the join with per-point
// counts, their exclusive scan into pair offsets, the total read back (synchronises the stream), then
// outputs(total, &lhs, &rhs) provides two device arrays of `total` elements, or leaves them NULL when no pairs are to be
// written, and k_pip_pairs fills them.
template <typename Outputs>
static int contains_pairs(gpl_ctx *ctx, const gpl_pip_index *idx, const double *pts, const uint8_t *validity, int64_t n,
                          Outputs outputs) {
    Scratch<int32_t> ids, cnt;
    Scratch<int64_t> off;
    GPL_TRY(ids.get(ctx, (size_t)n));
    GPL_TRY(cnt.get(ctx, (size_t)n));
    GPL_TRY(off.get(ctx, (size_t)n + 2));
    GPL_TRY(pip_query(ctx, idx, pts, validity, n, ids.p, cnt.p, ctx->stream));
    GPL_TRY((exclusive_scan<int32_t, int64_t>(ctx, cnt.p, n, off.p, off.p + n + 1)));
    int64_t total = 0;
    GPL_CUDA(cudaMemcpyAsync(&total, off.p + n + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    uint64_t *lhs = nullptr, *rhs = nullptr;
    GPL_TRY(outputs(total, &lhs, &rhs));
    if (lhs == nullptr) return GPL_OK;
    k_pip_pairs<<<pairs_grid(n), kQueryThreads, 0, ctx->stream>>>(view_of(idx), reinterpret_cast<const double2 *>(pts), validity, n,
                                                                  off.p, lhs, rhs);
    ctx->launches++;
    GPL_CUDA(cudaGetLastError());
    return GPL_OK;
}

extern "C" int gpl_contains_join_pairs(gpl_ctx *ctx, const gpl_pip_index *idx, const double *points_xy, int64_t n_points,
                                       uint64_t *lhs, uint64_t *rhs, int64_t *n_pairs, int mem) {
    GPL_REQUIRE(ctx && idx && n_pairs, GPL_ERR_INVALID_ARG, "gpl_contains_join_pairs: NULL argument");
    GPL_CUDA(cudaSetDevice(ctx->device));
    if (n_points == 0) {
        *n_pairs = 0;
        return GPL_OK;
    }
    Scratch<double> pts;
    const double *pdev = points_xy;
    if (mem == GPL_HOST) {
        GPL_TRY(pts.get(ctx, (size_t)n_points * 2));
        GPL_CUDA(cudaMemcpyAsync(pts.p, points_xy, sizeof(double) * 2 * n_points, cudaMemcpyHostToDevice, ctx->stream));
        pdev = pts.p;
    }
    const bool count_only = lhs == nullptr || rhs == nullptr;
    Scratch<uint64_t> dl, dr;
    GPL_TRY(contains_pairs(ctx, idx, pdev, nullptr, n_points, [&](int64_t total, uint64_t **pl, uint64_t **pr) -> int {
        if (!count_only)
            GPL_REQUIRE(*n_pairs >= total, GPL_ERR_INVALID_ARG, "pair buffers too small: need %lld, have %lld", (long long)total,
                        (long long)*n_pairs);
        *n_pairs = total;
        if (count_only || total == 0) return GPL_OK;
        *pl = lhs, *pr = rhs;
        if (mem == GPL_HOST) {
            GPL_TRY(dl.get(ctx, (size_t)total));
            GPL_TRY(dr.get(ctx, (size_t)total));
            *pl = dl.p, *pr = dr.p;
        }
        return GPL_OK;
    }));
    if (dl.p) {
        GPL_CUDA(cudaMemcpyAsync(lhs, dl.p, sizeof(uint64_t) * *n_pairs, cudaMemcpyDeviceToHost, ctx->stream));
        GPL_CUDA(cudaMemcpyAsync(rhs, dr.p, sizeof(uint64_t) * *n_pairs, cudaMemcpyDeviceToHost, ctx->stream));
    }
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    return GPL_OK;
}

// result of a join: defined in k_pairs.cu (gpl_spatial_join); the points-in-polygons join can return the same object
struct gpl_pairs {
    gpl_ctx *ctx = nullptr;
    uint64_t *lhs = nullptr, *rhs = nullptr;  // device
    int64_t n = 0;
};
extern "C" int gpl_contains_join_pairs_array(gpl_ctx *ctx, const gpl_pip_index *idx, const gpl_array *points, gpl_pairs **out) {
    GPL_REQUIRE(ctx && idx && points && out, GPL_ERR_INVALID_ARG, "gpl_contains_join_pairs_array: NULL argument");
    GPL_REQUIRE(points->type == GPL_POINT, GPL_ERR_INVALID_TYPE, "Expected Point (found geometry type %d)", points->type);
    GPL_CUDA(cudaSetDevice(ctx->device));
    gpl_pairs *res = new gpl_pairs();
    res->ctx = ctx;
    *out = res;
    const int64_t n = points->n_geoms;
    if (n == 0) return GPL_OK;
    GPL_TRY(contains_pairs(ctx, idx, points->xy, points->validity, n, [&](int64_t total, uint64_t **pl, uint64_t **pr) -> int {
        if (total == 0) return GPL_OK;
        void *l = nullptr, *r = nullptr;
        GPL_TRY(ctx->alloc(sizeof(uint64_t) * (size_t)total, &l));
        res->lhs = (uint64_t *)l;
        GPL_TRY(ctx->alloc(sizeof(uint64_t) * (size_t)total, &r));
        res->rhs = (uint64_t *)r;
        res->n = total;
        *pl = res->lhs, *pr = res->rhs;
        return GPL_OK;
    }));
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    return GPL_OK;
}

// End-to-end path: host points -> HBM -> ids -> host, chunked and double buffered so that the H2D of
// chunk k+1, the kernel of chunk k and the D2H of chunk k-1 overlap (PCIe Gen5 is full duplex).
extern "C" int gpl_contains_join_host(gpl_ctx *ctx, const gpl_pip_index *idx, const double *points_xy_host, int64_t n_points,
                                      int32_t *first_id_host, int64_t chunk_points) {
    GPL_REQUIRE(ctx && idx && (n_points == 0 || (points_xy_host && first_id_host)), GPL_ERR_INVALID_ARG,
                "gpl_contains_join_host: NULL argument");
    GPL_CUDA(cudaSetDevice(ctx->device));
    if (n_points == 0) return GPL_OK;
    if (chunk_points <= 0) chunk_points = 4 << 20;  // 64 MiB of points per chunk
    if (chunk_points > n_points) chunk_points = n_points;
    if (!ctx->copy_in) GPL_CUDA(cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking));
    if (!ctx->copy_out) GPL_CUDA(cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking));
    constexpr int NBUF = 3;
    Scratch<double> pts[NBUF];
    Scratch<int32_t> ids[NBUF];
    cudaEvent_t in_done[NBUF], k_done[NBUF], out_done[NBUF];
    for (int b = 0; b < NBUF; ++b) {
        GPL_TRY(pts[b].get(ctx, (size_t)chunk_points * 2));
        GPL_TRY(ids[b].get(ctx, (size_t)chunk_points));
        GPL_CUDA(cudaEventCreateWithFlags(&in_done[b], cudaEventDisableTiming));
        GPL_CUDA(cudaEventCreateWithFlags(&k_done[b], cudaEventDisableTiming));
        GPL_CUDA(cudaEventCreateWithFlags(&out_done[b], cudaEventDisableTiming));
    }
    // the scratch blocks may have been used by earlier work on ctx->stream: order the copy streams after it
    cudaEvent_t start;
    GPL_CUDA(cudaEventCreateWithFlags(&start, cudaEventDisableTiming));
    GPL_CUDA(cudaEventRecord(start, ctx->stream));
    GPL_CUDA(cudaStreamWaitEvent(ctx->copy_in, start, 0));
    GPL_CUDA(cudaStreamWaitEvent(ctx->copy_out, start, 0));
    int rc = GPL_OK;
    int64_t n_chunks = ceil_div(n_points, chunk_points);
    for (int64_t c = 0; c < n_chunks && rc == GPL_OK; ++c) {
        int b = (int)(c % NBUF);
        int64_t lo = c * chunk_points, n = std::min(chunk_points, n_points - lo);
        if (c >= NBUF) {
            cudaStreamWaitEvent(ctx->copy_in, k_done[b], 0);    // points buffer free once its kernel ran
            cudaStreamWaitEvent(ctx->stream, out_done[b], 0);   // ids buffer free once its D2H ran
        }
        cudaMemcpyAsync(pts[b].p, points_xy_host + 2 * lo, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, ctx->copy_in);
        cudaEventRecord(in_done[b], ctx->copy_in);
        cudaStreamWaitEvent(ctx->stream, in_done[b], 0);
        rc = pip_query(ctx, idx, pts[b].p, nullptr, n, ids[b].p, nullptr, ctx->stream);
        cudaEventRecord(k_done[b], ctx->stream);
        cudaStreamWaitEvent(ctx->copy_out, k_done[b], 0);
        cudaMemcpyAsync(first_id_host + lo, ids[b].p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->copy_out);
        cudaEventRecord(out_done[b], ctx->copy_out);
    }
    cudaError_t e1 = cudaStreamSynchronize(ctx->copy_out);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    cudaError_t e3 = cudaStreamSynchronize(ctx->copy_in);
    for (int b = 0; b < NBUF; ++b) {
        cudaEventDestroy(in_done[b]);
        cudaEventDestroy(k_done[b]);
        cudaEventDestroy(out_done[b]);
    }
    cudaEventDestroy(start);
    if (rc != GPL_OK) return rc;
    GPL_CUDA(e1);
    GPL_CUDA(e2);
    GPL_CUDA(e3);
    return GPL_OK;
}

extern "C" int gpl_join_histogram(gpl_ctx *ctx, const int32_t *first_id, int64_t n_points, uint64_t *counts, int64_t n_polygons,
                                  int mem) {
    GPL_REQUIRE(ctx && counts && (first_id || n_points == 0), GPL_ERR_INVALID_ARG, "gpl_join_histogram: NULL argument");
    GPL_REQUIRE(mem == GPL_DEVICE, GPL_ERR_UNSUPPORTED, "gpl_join_histogram: device buffers only");
    GPL_CUDA(cudaSetDevice(ctx->device));
    if (n_points == 0) return GPL_OK;
    GPL_TRY(launch_histogram(ctx, first_id, n_points, reinterpret_cast<unsigned long long *>(counts), n_polygons, ctx->stream));
    GPL_CUDA(cudaGetLastError());
    return GPL_OK;
}

