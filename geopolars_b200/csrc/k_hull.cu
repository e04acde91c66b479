// k_hull.cu — GeoSeries::convex_hull (reference: geopolars/geopolars-geo/src/geoseries.rs:23-26, impl `todo!()`
// at :196-198; py accessor py-geopolars/python/geopolars/internals/georust/geoseries.py:76-90).
// Arithmetic restated from geo 0.27 convex_hull/{mod,qhull}.rs (recalled, see oracle/geo_oracle.c):
//   hull = quick_hull(exterior coords incl. the closing duplicate); strict-CCW tests with the exact
//   orient2d; farthest point by p_orth . (p - a) evaluated in f64 with separately rounded mul/add;
//   output ring = [lower chain left->right, max, upper chain right->left, min, first again].
//
// B200 design: one warp per geometry.  The geometry's exterior coordinates are staged once into shared
// memory (coalesced LDG.128), permuted in place there exactly like geo permutes its Vec, and the
// recursion hull_set(a, b, slice) runs as an explicit stack machine whose control flow is warp-uniform:
//   * farthest point: lanes stride over the slice, warp arg-max (value, then LAST index: Iterator::max_by);
//   * partition by is_ccw: lanes evaluate the exact predicate for 32 elements at a time; __ballot_sync + popc
//     ranks reproduce geo's in-place Hoare partition as a set of disjoint swaps;
//   * the second recursive call is a tail call, so a frame is pushed only for the first one.
// Output rings have data-dependent length: pass 1 counts vertices per geometry, an exclusive scan turns
// counts into ring offsets, pass 2 re-runs the same deterministic machine and writes coordinates.
// Parity note: the slice permutations (swap_remove_to_first, the Hoare partition_slice) are reproduced element
// for element, so even exact ties for "farthest" resolve like the restated geo code (Iterator::max_by keeps the
// LAST maximal element of the slice).  DESIGN.md "convex_hull".
#include <math.h>

#include "common.cuh"
#include "scan.cuh"

namespace gpl {

constexpr int kHullWarps = 4;  // warps per CTA

struct HullFrame {  // pending "emit far, then hull_set(a, far, slice)" after the first recursive call returns
    double ax, ay;
    int32_t start, len, far_pos, pad;
};

__device__ __forceinline__ bool lex_less(double2 a, double2 b) { return a.x < b.x || (a.x == b.x && a.y < b.y); }
static __device__ __noinline__ double orient2d_noinline(double2 a, double2 b, double2 c) { return orient2d(a.x, a.y, b.x, b.y, c.x, c.y); }
static __device__ __noinline__ bool is_ccw_exact(double2 a, double2 b, double2 c) { return orient2d(a.x, a.y, b.x, b.y, c.x, c.y) > 0.0; }
// strict-CCW test.  The stage-A filter decides almost every call inline; only an uncertified determinant takes
// the out-of-line adaptive predicate (keeps the hot loops small: 122 -> ~80 registers).
__device__ __forceinline__ bool is_ccw(double2 a, double2 b, double2 c) {
    const double dl = (a.x - c.x) * (b.y - c.y);
    const double dr = (a.y - c.y) * (b.x - c.x);
    const double det = dl - dr;
    if (fabs(det) > kCcwA * (fabs(dl) + fabs(dr))) return det > 0.0;
    return is_ccw_exact(a, b, c);
}

// geo's utils::partition_slice on P[s, s+len) with predicate is_ccw(a, b, .): an in-place Hoare scheme
//     loop { while l < len && pred(l) { l++ }  while r > 0 && !pred(r) { r-- }  if l >= r { return l }  swap(l, r) }
// whose result is fully determined by the predicate bits: with T = number of trues, the i-th FALSE element
// (ascending) among positions < T is swapped with the i-th TRUE element counted from the right among
// positions >= T; every other element stays where it is.  That is what the warp does: predicate ballots
// (one exact orient2d per element), ranks from popc prefix counts, the two position lists in scratch, then
// disjoint pairwise swaps.  The slice order therefore equals geo's element for element, which matters only
// for the arg-max tie rule of hull_set.  `scratch` holds at least len int32 (it is the tmp buffer).
// Returns T.
__device__ __forceinline__ int32_t partition_ccw(double2 *P, double2 *tmp, int32_t s, int32_t len, double2 a, double2 b, int lane) {
    if (len <= 0) return 0;
    int32_t *scratch = reinterpret_cast<int32_t *>(tmp);  // [0, len): left-false positions, [len, 2 len): right-true positions
    unsigned *masks = reinterpret_cast<unsigned *>(scratch + 2 * len);  // one ballot per 32 elements
    const unsigned below = (1u << lane) - 1u;
    int32_t n_true = 0;
    for (int32_t c = 0; c < len; c += 32) {
        const int32_t i = c + lane;
        const bool t = i < len && is_ccw(a, b, P[s + i]);
        const unsigned mt = __ballot_sync(0xffffffffu, t);
        if (lane == 0) masks[c >> 5] = mt;
        n_true += __popc(mt);
    }
    __syncwarp();
    const int32_t T = n_true;
    int32_t trues_before = 0;
    for (int32_t c = 0; c < len; c += 32) {
        const int32_t i = c + lane;
        const unsigned mt = masks[c >> 5];
        const bool in = i < len, t = (mt >> lane) & 1u;
        const int32_t tb = trues_before + __popc(mt & below);  // trues in [0, i)
        if (in && !t && i < T) scratch[i - tb] = i;                       // rank among left falses = falses in [0, i)
        if (in && t && i >= T) scratch[len + (T - tb - 1)] = i;           // rank from the right = trues in (i, len)
        trues_before += __popc(mt);
    }
    __syncwarp();
    // number of misplaced pairs = falses among the first T positions
    int32_t falses_left = 0;
    for (int32_t c = 0; c < T; c += 32) {
        const unsigned mt = masks[c >> 5];
        const int32_t width = min(32, T - c);
        const unsigned valid = width == 32 ? 0xffffffffu : ((1u << width) - 1u);
        falses_left += __popc(~mt & valid);
    }
    for (int32_t i = lane; i < falses_left; i += 32) {
        const int32_t f = scratch[i], t = scratch[len + i];
        const double2 x = P[s + f];
        P[s + f] = P[s + t];
        P[s + t] = x;
    }
    __syncwarp();
    return T;
}

// index (within the slice) of the farthest point from segment a-b: max of p_orth . (p - a), LAST maximal element
__device__ __forceinline__ int32_t farthest(const double2 *P, int32_t s, int32_t len, double2 a, double2 b, int lane) {
    const double ox = a.y - b.y, oy = b.x - a.x;
    double best = 0.0;
    int32_t bi = -1;
    for (int32_t i = lane; i < len; i += 32) {
        const double2 q = P[s + i];
        const double dx = q.x - a.x, dy = q.y - a.y;
        const double v = ox * dx + oy * dy;
        if (bi < 0 || !(v < best)) {  // max_by keeps the later element on ties
            best = v;
            bi = i;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int32_t oi = __shfl_xor_sync(0xffffffffu, bi, o);
        // lanes hold disjoint index sets: take the other if it is strictly better, or equal with a later index
        const bool take = oi >= 0 && (bi < 0 || ov > best || (!(ov < best) && oi > bi));
        if (take) {
            best = ov;
            bi = oi;
        }
    }
    return bi;
}

template <bool WRITE>
struct Emitter {
    double2 *out;
    int64_t n;
    double2 first;
    __device__ __forceinline__ void push(double2 p, int lane) {
        if (n == 0) first = p;
        if (WRITE && lane == 0) out[n] = p;
        ++n;
    }
};

// geo trivial_hull(points, include_on_hull = false) for fewer than four coordinates (lane-uniform, tiny)
template <bool WRITE>
__device__ __forceinline__ void trivial_hull(const double2 *P, int32_t n, Emitter<WRITE> &em, int lane) {
    double2 ls[4];
    int32_t m = n;
    for (int32_t i = 0; i < n; ++i) ls[i] = P[i];
    for (int32_t i = 1; i < m; ++i)  // sort_unstable_by(lex_cmp) on <= 3 items: any correct sort gives the same result
        for (int32_t j = i; j > 0 && lex_less(ls[j], ls[j - 1]); --j) {
            double2 t = ls[j];
            ls[j] = ls[j - 1];
            ls[j - 1] = t;
        }
    if (m == 3 && orient2d(ls[0].x, ls[0].y, ls[1].x, ls[1].y, ls[2].x, ls[2].y) == 0.0) {
        ls[1] = ls[2];
        m = 2;
    }
    if (m == 0) return;
    if (m == 1) ls[m++] = ls[0];
    if (!(ls[0].x == ls[m - 1].x && ls[0].y == ls[m - 1].y)) ls[m++] = ls[0];  // close
    if (m >= 4) {  // make_ccw_winding: least index is 0 after the sort, prev = m-2, next = 1
        if (orient2d(ls[m - 2].x, ls[m - 2].y, ls[0].x, ls[0].y, ls[1].x, ls[1].y) < 0.0) {
            double2 t = ls[1];  // reverse [p0,p1,p2,p0] -> [p0,p2,p1,p0]
            ls[1] = ls[m - 2];
            ls[m - 2] = t;
        }
    }
    for (int32_t i = 0; i < m; ++i) em.push(ls[i], lane);
}

// hull_set(a, b, P[s, s+len)) as a stack machine; emits vertices in geo's order
template <bool WRITE>
__device__ __forceinline__ void hull_set(double2 *P, double2 *tmp, HullFrame *stack, double2 a, double2 b, int32_t s, int32_t len,
                                         Emitter<WRITE> &em, int lane) {
    int32_t depth = 0;
    for (;;) {
        if (len >= 2) {
            const int32_t fi = farthest(P, s, len, a, b, lane);
            if (lane == 0) {  // swap_remove_to_first
                double2 t = P[s];
                P[s] = P[s + fi];
                P[s + fi] = t;
            }
            __syncwarp();
            const double2 far = P[s];
            const int32_t s1 = s + 1, l1 = len - 1;
            const int32_t k = partition_ccw(P, tmp, s1, l1, far, b, lane);
            if (lane == 0) {
                HullFrame f;
                f.ax = a.x, f.ay = a.y, f.start = s1, f.len = l1, f.far_pos = s, f.pad = 0;
                stack[depth] = f;
            }
            __syncwarp();
            ++depth;
            a = far;  // hull_set(far, b, P[s1, s1+k))
            s = s1;
            len = k;
            continue;
        }
        if (len == 1) em.push(P[s], lane);
        if (depth == 0) return;
        --depth;
        const HullFrame f = stack[depth];
        const double2 far = P[f.far_pos];
        em.push(far, lane);
        const double2 fa = make_double2(f.ax, f.ay);
        const int32_t k2 = partition_ccw(P, tmp, f.start, f.len, fa, far, lane);
        a = fa;  // tail call hull_set(a, far, P[start, start+k2))
        b = far;
        s = f.start;
        len = k2;
    }
}

// number of exterior coordinates of geometry g and a gather of them into dst (CoordsIter::exterior_coords_iter)
__device__ __forceinline__ int64_t exterior_count(int type, int64_t g, const int64_t *geom_off, const int64_t *part_off,
                                                  const int64_t *ring_off) {
    switch (type) {
    case GPL_POINT: return 1;
    case GPL_LINESTRING:
    case GPL_MULTIPOINT: return geom_off[g + 1] - geom_off[g];
    case GPL_MULTILINESTRING: return ring_off[geom_off[g + 1]] - ring_off[geom_off[g]];
    case GPL_POLYGON: return geom_off[g + 1] > geom_off[g] ? ring_off[geom_off[g] + 1] - ring_off[geom_off[g]] : 0;
    default: {
        int64_t n = 0;
        for (int64_t p = geom_off[g]; p < geom_off[g + 1]; ++p)
            if (part_off[p + 1] > part_off[p]) n += ring_off[part_off[p] + 1] - ring_off[part_off[p]];
        return n;
    }
    }
}
__device__ __forceinline__ void exterior_gather(int type, int64_t g, const double2 *__restrict__ xy, const int64_t *geom_off,
                                                const int64_t *part_off, const int64_t *ring_off, double2 *dst, int lane) {
    int64_t c0 = 0, c1 = 0;
    switch (type) {
    case GPL_POINT: c0 = g, c1 = g + 1; break;
    case GPL_LINESTRING:
    case GPL_MULTIPOINT: c0 = geom_off[g], c1 = geom_off[g + 1]; break;
    case GPL_MULTILINESTRING: c0 = ring_off[geom_off[g]], c1 = ring_off[geom_off[g + 1]]; break;
    case GPL_POLYGON:
        if (geom_off[g + 1] > geom_off[g]) c0 = ring_off[geom_off[g]], c1 = ring_off[geom_off[g] + 1];
        break;
    default: {
        int64_t o = 0;
        for (int64_t p = geom_off[g]; p < geom_off[g + 1]; ++p) {
            if (part_off[p + 1] <= part_off[p]) continue;
            const int64_t a = ring_off[part_off[p]], b = ring_off[part_off[p] + 1];
            for (int64_t c = a + lane; c < b; c += 32) dst[o + (c - a)] = __ldcs(xy + c);
            o += b - a;
        }
        return;
    }
    }
    for (int64_t c = c0 + lane; c < c1; c += 32) dst[c - c0] = __ldcs(xy + c);
}

// max exterior coordinate count over all geometries (sizes the per-warp staging area)
__global__ void k_hull_max_len(int type, int64_t n_geoms, const int64_t *__restrict__ geom_off, const int64_t *__restrict__ part_off,
                               const int64_t *__restrict__ ring_off, unsigned long long *__restrict__ out) {
    int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    unsigned long long v = 0;
    if (g < n_geoms) v = (unsigned long long)exterior_count(type, g, geom_off, part_off, ring_off);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long t = __shfl_xor_sync(0xffffffffu, v, o);
        v = t > v ? t : v;
    }
    if ((threadIdx.x & 31) == 0 && v) atomicMax(out, v);
}

// One warp per geometry.  The staging area (points + partition scratch) is in shared memory when the largest
// geometry fits (SMEM = true: the pointers are derived from the __shared__ array only, so the compiler emits
// LDS/STS instead of generic loads), otherwise in a per-warp global workspace.  The frame stack (one push
// and one pop per hull_set call) always lives in the global workspace.
template <bool WRITE, bool SMEM>
__global__ void __launch_bounds__(kHullWarps * 32, SMEM ? 5 : 2) k_hull(int type, int64_t n_geoms, const double2 *__restrict__ xy,
                                                                        const int64_t *__restrict__ geom_off,
                                                                        const int64_t *__restrict__ part_off,
                                                                        const int64_t *__restrict__ ring_off,
                                                                        const uint8_t *__restrict__ validity, int32_t cap,
                                                                        uint8_t *__restrict__ workspace, int64_t *__restrict__ counts,
                                                                        const int64_t *__restrict__ out_off, double2 *__restrict__ out_xy,
                                                                        const uint8_t *__restrict__ only) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const size_t warp_slot = (size_t)blockIdx.x * kHullWarps + wid;
    const size_t stack_bytes = (size_t)cap * sizeof(HullFrame), stage_bytes = (size_t)cap * 2 * sizeof(double2);
    HullFrame *stack = reinterpret_cast<HullFrame *>(workspace + warp_slot * (stack_bytes + (SMEM ? 0 : stage_bytes)));
    double2 *P, *tmp;
    if (SMEM) {
        P = reinterpret_cast<double2 *>(smem) + (size_t)wid * 2 * cap;
    } else {
        P = reinterpret_cast<double2 *>(workspace + warp_slot * (stack_bytes + stage_bytes) + stack_bytes);
    }
    tmp = P + cap;
    const int64_t n_warps = (int64_t)gridDim.x * kHullWarps;
    for (int64_t g = (int64_t)blockIdx.x * kHullWarps + wid; g < n_geoms; g += n_warps) {
        if (!only[g]) continue;  // the level-wise kernel finished this geometry
        Emitter<WRITE> em;
        em.n = 0;
        em.out = WRITE ? out_xy + out_off[g] : nullptr;
        em.first = make_double2(0.0, 0.0);
        if (bit_get(validity, g)) {
            int32_t n = (int32_t)exterior_count(type, g, geom_off, part_off, ring_off);
            __syncwarp();
            exterior_gather(type, g, xy, geom_off, part_off, ring_off, P, lane);
            __syncwarp();
            if (n < 4) {
                trivial_hull<WRITE>(P, n, em, lane);
            } else {
                // utils::least_and_greatest_index: FIRST least and FIRST greatest in lexicographic order
                int32_t mi = -1, xi = -1;
                double2 mn = make_double2(0.0, 0.0), mx = mn;
                for (int32_t i = lane; i < n; i += 32) {
                    const double2 q = P[i];
                    if (mi < 0 || lex_less(q, mn)) mn = q, mi = i;
                    if (xi < 0 || lex_less(mx, q)) mx = q, xi = i;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ox = __shfl_xor_sync(0xffffffffu, mn.x, o), oy = __shfl_xor_sync(0xffffffffu, mn.y, o);
                    const int32_t oi = __shfl_xor_sync(0xffffffffu, mi, o);
                    const double2 oq = make_double2(ox, oy);
                    if (oi >= 0 && (mi < 0 || lex_less(oq, mn) || (!lex_less(mn, oq) && oi < mi))) mn = oq, mi = oi;
                    const double px = __shfl_xor_sync(0xffffffffu, mx.x, o), py = __shfl_xor_sync(0xffffffffu, mx.y, o);
                    const int32_t pi = __shfl_xor_sync(0xffffffffu, xi, o);
                    const double2 pq = make_double2(px, py);
                    if (pi >= 0 && (xi < 0 || lex_less(mx, pq) || (!lex_less(pq, mx) && pi < xi))) mx = pq, xi = pi;
                }
                int32_t min_idx = mi, max_idx = xi;
                if (lane == 0) {  // swap_remove_to_first(min), then fix up max_idx exactly like geo
                    double2 t = P[0];
                    P[0] = P[min_idx];
                    P[min_idx] = t;
                }
                __syncwarp();
                if (max_idx == 0) max_idx = min_idx;
                max_idx = max_idx > 0 ? max_idx - 1 : 0;
                if (lane == 0) {
                    double2 t = P[1];
                    P[1] = P[1 + max_idx];
                    P[1 + max_idx] = t;
                }
                __syncwarp();
                const double2 pmin = P[0], pmax = P[1];
                const int32_t s = 2, len = n - 2;
                int32_t k = partition_ccw(P, tmp, s, len, pmax, pmin, lane);
                hull_set<WRITE>(P, tmp, stack, pmax, pmin, s, k, em, lane);
                em.push(pmax, lane);
                k = partition_ccw(P, tmp, s, len, pmin, pmax, lane);
                hull_set<WRITE>(P, tmp, stack, pmin, pmax, s, k, em, lane);
                em.push(pmin, lane);
                if (!(em.first.x == pmin.x && em.first.y == pmin.y)) em.push(em.first, lane);  // LineString::close
            }
        }
        if (counts != nullptr && lane == 0) counts[g] = em.n;
        __syncwarp();
    }
}

// ---- fast path: the same recursion, level by level -----------------------------------------------------------------
// geo's quick_hull is a depth-first recursion over ever smaller slices; run by one warp it spends most of its ~11 k
// instructions on slices of a handful of points (3 of 32 lanes busy) and on the warp-wide bookkeeping of each of its ~50 calls.
// The recursion TREE, however, does not depend on the order in which the calls are made: a call hull_set(a, b, S) picks
// far = argmax over S of orth(a,b) . (p - a) (evaluated in f64 exactly like geo) and splits S \ {far} into
// {p : ccw(far, b, p)} and {p : ccw(a, far, p)} — functions of (a, b, S) alone.  The only place where geo's slice ORDER
// matters is the arg-max tie rule (Iterator::max_by keeps the last maximal element of the slice as permuted by the Hoare
// partitions).  So: process all calls of one recursion depth together (every live point carries the id of its call; the
// warp's lanes stride over the live points, whatever call they belong to), and whenever two points with DIFFERENT
// coordinates tie for a maximum — or anything else happens that the level-wise form does not cover (non-finite coordinates,
// fewer than four coordinates, min == max, a point that is strictly left of both child segments, more than 128 calls alive)
// — flag the geometry and let the order-exact kernel above redo it.  Points with EQUAL coordinates tying (the closing
// duplicate of a ring is one in every polygon) do not matter: whichever copy is taken, the others are collinear with
// every segment through it and are dropped by both partitions, as in geo.
// The emission order of geo (lower chain from min towards max, max, upper chain back, min, closing copy of the first) is
// kept as a CHAIN of vertex ids in emission order; the points of a call sit "before" the chain vertex that is the call's
// `a`, with `b` the previous chain vertex (cyclically); a call's far point is inserted before its `a`.
constexpr int kHullSegCap = 128;  // live calls per level (chain length); beyond it the geometry is redone by k_hull
struct HullFastLayout {
    // per warp, in shared memory: P0[cap] double2 | KV[cap] u64 | EA[cap] u32 | EB[cap] u32 | HI[S] u32 | LO[S] u32 | FAR[S] i32 |
    // NI[S] i32 | CHA[S] u16 | CHB[S] u16
    static __host__ __device__ size_t bytes(int cap) { return (size_t)cap * 32 + (size_t)kHullSegCap * 20; }
};
__device__ __forceinline__ unsigned long long hull_ord(double d) {  // order-preserving, > 0 for every non-NaN value
    const unsigned long long b = (unsigned long long)__double_as_longlong(d);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
template <bool WRITE>
__global__ void __launch_bounds__(kHullWarps * 32, 5) k_hull_fast(int type, int64_t n_geoms, const double2 *__restrict__ xy,
                                                               const int64_t *__restrict__ geom_off, const int64_t *__restrict__ part_off,
                                                               const int64_t *__restrict__ ring_off, const uint8_t *__restrict__ validity,
                                                               int32_t cap, int64_t *__restrict__ counts, const int64_t *__restrict__ out_off,
                                                               double2 *__restrict__ out_xy, uint8_t *__restrict__ redo) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint8_t *base = smem + (size_t)wid * HullFastLayout::bytes(cap);
    double2 *P0 = reinterpret_cast<double2 *>(base);
    unsigned long long *KV = reinterpret_cast<unsigned long long *>(base + (size_t)cap * 16);  // this level's key of every live point
    uint32_t *EA = reinterpret_cast<uint32_t *>(base + (size_t)cap * 24), *EB = EA + cap;
    uint32_t *HI = EB + cap, *LO = HI + kHullSegCap;
    int32_t *FAR = reinterpret_cast<int32_t *>(LO + kHullSegCap), *NI = FAR + kHullSegCap;
    uint16_t *CHA = reinterpret_cast<uint16_t *>(NI + kHullSegCap), *CHB = CHA + kHullSegCap;
    const unsigned below = (1u << lane) - 1u;
    const int64_t n_warps = (int64_t)gridDim.x * kHullWarps;
    for (int64_t g = (int64_t)blockIdx.x * kHullWarps + wid; g < n_geoms; g += n_warps) {
        bool flag = false;       // warp-uniform: redo this geometry with the order-exact kernel
        int64_t n_out = 0;
        if (bit_get(validity, g)) {
            const int64_t n64 = exterior_count(type, g, geom_off, part_off, ring_off);
            if (n64 < 4 || n64 > cap) {
                flag = true;
            } else {
                const int32_t n = (int32_t)n64;
                __syncwarp();
                exterior_gather(type, g, xy, geom_off, part_off, ring_off, P0, lane);
                __syncwarp();
                // ---- lexicographic min / max (any instance: equal coordinates are interchangeable here), finiteness
                int32_t mi = -1, xi = -1;
                double2 mn = make_double2(0.0, 0.0), mx = mn;
                bool bad = false;
                for (int32_t i = lane; i < n; i += 32) {
                    const double2 q = P0[i];
                    bad = bad || !(isfinite(q.x) && isfinite(q.y));
                    if (mi < 0 || lex_less(q, mn)) mn = q, mi = i;
                    if (xi < 0 || lex_less(mx, q)) mx = q, xi = i;
                }
                // warp arg-min / arg-max of (x, then y, then lowest index) through REDUX on order-preserving keys: the 5-step
                // butterfly over (x, y, index) cost ~250 instructions per polygon.  x + 0.0 maps -0.0 to +0.0 (equal as doubles).
                {
                    auto warp_pick = [&](bool want_max, double2 &v, int32_t &vi) {
                        unsigned cand = __ballot_sync(0xffffffffu, vi >= 0);
                        const double ord[2] = {v.x + 0.0, v.y + 0.0};
#pragma unroll
                        for (int d = 0; d < 2 && __popc(cand) > 1; ++d) {
                            unsigned long long k = hull_ord(ord[d]);
                            if (want_max) k = ~k;  // arg-max as arg-min of the complement
                            const bool in = (cand >> lane) & 1u;
                            const uint32_t h = __reduce_min_sync(0xffffffffu, in ? (uint32_t)(k >> 32) : 0xffffffffu);
                            const bool c1 = in && (uint32_t)(k >> 32) == h;
                            const uint32_t l = __reduce_min_sync(0xffffffffu, c1 ? (uint32_t)k : 0xffffffffu);
                            cand = __ballot_sync(0xffffffffu, c1 && (uint32_t)k == l);
                        }
                        if (__popc(cand) > 1) {  // equal coordinates: the lowest index (any instance would do)
                            const bool in = (cand >> lane) & 1u;
                            const uint32_t i0 = __reduce_min_sync(0xffffffffu, in ? (uint32_t)vi : 0xffffffffu);
                            cand = __ballot_sync(0xffffffffu, in && (uint32_t)vi == i0);
                        }
                        const int src = __ffs(cand) - 1;  // n >= 4: at least one lane holds a point
                        v.x = __shfl_sync(0xffffffffu, v.x, src), v.y = __shfl_sync(0xffffffffu, v.y, src);
                        vi = __shfl_sync(0xffffffffu, vi, src);
                    };
                    warp_pick(false, mn, mi);
                    warp_pick(true, mx, xi);
                }
                flag = __any_sync(0xffffffffu, bad) || (mn.x == mx.x && mn.y == mx.y);
                int32_t m = 2, ne = 0;  // chain length, live points
                uint32_t *E = EA, *En = EB;
                uint16_t *CH = CHA, *CHn = CHB;
                if (!flag) {
                    if (lane == 0) CH[0] = (uint16_t)xi, CH[1] = (uint16_t)mi;  // emission order: [.., max, .., min]
                    // ---- level 0: strictly right of min->max (= left of max->min) is the lower set (call 0), strictly left the upper (call 1)
                    for (int32_t c = 0; c < n; c += 32) {
                        const int32_t i = c + lane;
                        int side = 0;
                        if (i < n) {
                            const double2 q = P0[i];
                            const double dl = (mx.x - q.x) * (mn.y - q.y), dr = (mx.y - q.y) * (mn.x - q.x);
                            const double det = dl - dr;
                            if (fabs(det) > kCcwA * (fabs(dl) + fabs(dr))) side = det > 0.0 ? 1 : 2;
                            else {
                                const double ex = orient2d_noinline(mx, mn, q);
                                side = ex > 0.0 ? 1 : (ex < 0.0 ? 2 : 0);
                            }
                        }
                        const unsigned mk = __ballot_sync(0xffffffffu, side != 0);
                        if (side) E[ne + __popc(mk & below)] = (uint32_t)i | ((uint32_t)(side - 1) << 16);
                        ne += __popc(mk);
                    }
                    __syncwarp();
                }
                // ---- one iteration per recursion depth
                // zero the per-call maxima of the first `cnt` calls
                auto zero_calls = [&](int32_t cnt) {
                    for (int32_t j = lane; j < cnt; j += 32) HI[j] = 0u, LO[j] = 0u;
                    __syncwarp();
                };
                // A: per call, the maximum of orth(a,b) . (p - a): high word first.  Two rows of 32 points per round, all
                // loads of both rows issued before the first use (the chain E -> CH -> P0 is three dependent shared loads).
                auto pass_a = [&]() {
                    for (int32_t c = 0; c < ne; c += 64) {
                        uint32_t sgv[2], hiv[2];
                        unsigned long long kv[2];
                        bool inr[2];
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            const int32_t e = c + 32 * u + lane;
                            inr[u] = e < ne;
                            const uint32_t w = E[inr[u] ? e : 0];
                            sgv[u] = w >> 16;
                            const double2 p = P0[w & 0xffffu], a = P0[CH[sgv[u]]], b = P0[CH[sgv[u] ? sgv[u] - 1 : m - 1]];
                            const double ox = a.y - b.y, oy = b.x - a.x, dx = p.x - a.x, dy = p.y - a.y;
                            kv[u] = hull_ord(ox * dx + oy * dy);
                            hiv[u] = inr[u] ? (uint32_t)(kv[u] >> 32) : 0u;
                        }
#pragma unroll
                        for (int u = 0; u < 2; ++u)
                            if (inr[u]) KV[c + 32 * u + lane] = kv[u];
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            if (c + 32 * u >= ne) break;  // warp-uniform
                            const uint32_t sg0 = __shfl_sync(0xffffffffu, sgv[u], 0);
                            if (__all_sync(0xffffffffu, !inr[u] || sgv[u] == sg0)) {  // a whole row of one call: one atomic instead of 32 colliding ones
                                const uint32_t r = __reduce_max_sync(0xffffffffu, hiv[u]);
                                if (lane == 0) atomicMax(&HI[sg0], r);
                            } else if (inr[u]) {
                                atomicMax(&HI[sgv[u]], hiv[u]);
                            }
                        }
                    }
                    __syncwarp();
                };
                // B: the far point of every live call = the point holding the call's maximal key.  Returns true when two points
                // with different coordinates tie somewhere (geo's slice order would decide — not reproduced here).
                auto pass_b = [&]() -> bool {
                    // the points that hold their call's high word; one per call (nearly always): it is the far point
                    bool multi = false;
                    for (int32_t c = 0; c < ne; c += 32) {
                        const int32_t e = c + lane;
                        if (e < ne) {
                            const uint32_t w = E[e], sg = w >> 16;
                            if ((uint32_t)(KV[e] >> 32) == HI[sg]) {
                                multi = multi || atomicAdd(&LO[sg], 1u) > 0u;
                                FAR[sg] = (int32_t)(w & 0xffffu);
                            }
                        }
                    }
                    const bool any_multi = __any_sync(0xffffffffu, multi);
                    __syncwarp();
                    if (!any_multi) return false;
                    // several points share a high word somewhere: low word among them, then the holder(s) of the full key
                    for (int32_t j = lane; j < m; j += 32) LO[j] = 0u;
                    __syncwarp();
                    for (int32_t c = 0; c < ne; c += 32) {
                        const int32_t e = c + lane;
                        if (e < ne) {
                            const uint32_t sg = E[e] >> 16;
                            const unsigned long long k = KV[e];
                            if ((uint32_t)(k >> 32) == HI[sg]) atomicMax(&LO[sg], (uint32_t)k);
                        }
                    }
                    __syncwarp();
                    for (int32_t c = 0; c < ne; c += 32) {
                        const int32_t e = c + lane;
                        if (e < ne) {
                            const uint32_t w = E[e], sg = w >> 16;
                            const unsigned long long k = KV[e];
                            if ((uint32_t)(k >> 32) == HI[sg] && (uint32_t)k == LO[sg]) FAR[sg] = (int32_t)(w & 0xffffu);
                        }
                    }
                    __syncwarp();
                    bool tie = false;
                    for (int32_t c = 0; c < ne; c += 32) {
                        const int32_t e = c + lane;
                        if (e < ne) {
                            const uint32_t w = E[e], sg = w >> 16;
                            const unsigned long long k = KV[e];
                            if ((uint32_t)(k >> 32) == HI[sg] && (uint32_t)k == LO[sg]) {
                                const double2 p = P0[w & 0xffffu], f = P0[FAR[sg]];
                                tie = tie || !(p.x == f.x && p.y == f.y);
                            }
                        }
                    }
                    return __any_sync(0xffffffffu, tie);
                };
                while (!flag && ne > 0) {
                    zero_calls(m);
                    pass_a();
                    if (pass_b()) {
                        flag = true;
                        break;
                    }
                    // chain update: the far point of every live call goes in front of the call's `a`
                    int32_t added = 0;
                    for (int32_t c = 0; c < m; c += 32) {
                        const int32_t j = c + lane;
                        const bool live = j < m && HI[j] != 0u;
                        const unsigned mk = __ballot_sync(0xffffffffu, live);
                        if (j < m) {
                            const int32_t nj = j + added + __popc(mk & below) + (live ? 1 : 0);
                            NI[j] = nj;
                            if (nj < kHullSegCap) CHn[nj] = CH[j];
                            if (live && nj - 1 < kHullSegCap) CHn[nj - 1] = (uint16_t)FAR[j];
                        }
                        added += __popc(mk);
                    }
                    if (m + added > kHullSegCap) {
                        flag = true;
                        break;
                    }
                    __syncwarp();
                    // E: every point moves to one of its call's two children, or drops out (two rows per round, as in A).
                    // (Forming the child call's key here, from the coordinates already in registers, saves pass A's loads but
                    // measured slower: 33.0 vs 28.2 ms per 3 M polygons — more live registers, more spills.)
                    int32_t ne2 = 0;
                    bool both = false;
                    for (int32_t c = 0; c < ne; c += 64) {
                        uint32_t nw[2];
                        bool keep[2];
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            const int32_t e = c + 32 * u + lane;
                            const bool in = e < ne;
                            const uint32_t w = E[in ? e : 0], sg = w >> 16, pi = w & 0xffffu;
                            const int32_t nj = NI[sg];
                            const double2 p = P0[pi], a = P0[CH[sg]], b = P0[CH[sg ? sg - 1 : m - 1]], f = P0[FAR[sg]];
                            keep[u] = false, nw[u] = 0u;
                            if (in && !(p.x == f.x && p.y == f.y)) {
                                const bool t1 = is_ccw(f, b, p), t2 = is_ccw(a, f, p);
                                both = both || (t1 && t2);
                                keep[u] = t1 || t2;
                                nw[u] = pi | ((uint32_t)(t1 ? nj - 1 : nj) << 16);
                            }
                        }
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            const unsigned mk = __ballot_sync(0xffffffffu, keep[u]);
                            if (keep[u]) En[ne2 + __popc(mk & below)] = nw[u];
                            ne2 += __popc(mk);
                        }
                    }
                    if (__any_sync(0xffffffffu, both)) {
                        flag = true;
                        break;
                    }
                    __syncwarp();
                    {
                        uint32_t *t = E;
                        E = En, En = t;
                        uint16_t *u = CH;
                        CH = CHn, CHn = u;
                    }
                    m += added;
                    ne = ne2;
                }
                if (!flag) {  // the chain IS the ring: [.., max, .., min] (+ the closing copy of the first vertex)
                    const double2 first = P0[CH[0]];
                    const bool close = !(first.x == mn.x && first.y == mn.y);
                    n_out = m + (close ? 1 : 0);
                    if (WRITE) {
                        double2 *dst = out_xy + out_off[g];
                        for (int32_t j = lane; j < m; j += 32) dst[j] = P0[CH[j]];
                        if (close && lane == 0) dst[m] = first;
                    }
                }
            }
        }
        if (lane == 0) {
            if (redo) redo[g] = flag ? 1 : 0;
            if (counts != nullptr && !flag) counts[g] = n_out;
        }
        __syncwarp();
    }
}

// upper bound of the hull ring length of geometry g: all exterior coordinates + the closing vertex
__global__ void k_hull_upper(int type, int64_t n_geoms, const int64_t *__restrict__ geom_off, const int64_t *__restrict__ part_off,
                             const int64_t *__restrict__ ring_off, int64_t *__restrict__ ub) {
    int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g < n_geoms) ub[g] = exterior_count(type, g, geom_off, part_off, ring_off) + 2;
}
// one warp per geometry: move the ring from its slot in the temporary buffer to its final offset
__global__ void __launch_bounds__(256) k_hull_compact(int64_t n_geoms, const double2 *__restrict__ tmp, const int64_t *__restrict__ tmp_off,
                                                      const int64_t *__restrict__ out_off, double2 *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t g = warp; g < n_geoms; g += nwarps) {
        const int64_t s = tmp_off[g], d = out_off[g], m = out_off[g + 1] - d;
        for (int64_t k = lane; k < m; k += 32) out[d + k] = tmp[s + k];
    }
}
__global__ void k_iota(int64_t *__restrict__ out, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = i;
}

}  // namespace gpl

using namespace gpl;

extern "C" int gpl_convex_hull(gpl_ctx *ctx, const gpl_array *in, gpl_array **out) {
    GPL_REQUIRE(ctx && in && out, GPL_ERR_INVALID_ARG, "gpl_convex_hull: NULL argument");
    GPL_CUDA(cudaSetDevice(ctx->device));
    const int64_t n = in->n_geoms;
    const double2 *xy = reinterpret_cast<const double2 *>(in->xy);
    Scratch<unsigned long long> maxlen;
    Scratch<int64_t> counts, total;
    GPL_TRY(maxlen.get(ctx, 1));
    GPL_TRY(counts.get(ctx, (size_t)n + 1));
    GPL_TRY(total.get(ctx, 1));
    GPL_CUDA(cudaMemsetAsync(maxlen.p, 0, sizeof(unsigned long long), ctx->stream));
    if (n > 0) GPL_LAUNCH(ctx, k_hull_max_len, (int)ceil_div(n, 256), 256, 0, in->type, n, in->geom_off, in->part_off, in->ring_off, maxlen.p);
    unsigned long long h_max = 0;
    GPL_CUDA(cudaMemcpyAsync(&h_max, maxlen.p, sizeof(h_max), cudaMemcpyDeviceToHost, ctx->stream));
    GPL_CUDA(cudaStreamSynchronize(ctx->stream));
    GPL_REQUIRE(h_max < (1ULL << 30), GPL_ERR_UNSUPPORTED, "convex_hull: a geometry with %llu coordinates is too large", h_max);
    const int32_t cap = (int32_t)std::max<unsigned long long>(h_max, 4);
    const size_t stage_bytes = (size_t)cap * 2 * sizeof(double2), stack_bytes = (size_t)cap * sizeof(HullFrame);
    const size_t smem_bytes = stage_bytes * kHullWarps;
    const bool use_smem = smem_bytes <= 200 * 1024;
    int grid;
    Scratch<uint8_t> workspace;
    if (use_smem) {
        GPL_CUDA(cudaFuncSetAttribute(k_hull<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        GPL_CUDA(cudaFuncSetAttribute(k_hull<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        int per_sm = (int)std::max<size_t>(1, std::min<size_t>(5, (220 * 1024) / std::max<size_t>(smem_bytes, 1)));
        grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(std::max<int64_t>(n, 1), kHullWarps), (int64_t)kSMs * per_sm));
    } else {
        grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(std::max<int64_t>(n, 1), kHullWarps), (int64_t)kSMs * 2));
    }
    GPL_TRY(workspace.get(ctx, (stack_bytes + (use_smem ? 0 : stage_bytes)) * kHullWarps * (size_t)grid));
    const size_t dyn = use_smem ? smem_bytes : 0;
    // The level-wise kernel takes every geometry it can (4 <= coordinates <= fast_cap, finite, no arg-max tie between distinct
    // points); what it flags in `redo` is recomputed by the order-exact kernel.
    const int32_t fast_cap = (int32_t)((std::min<unsigned long long>(std::max<unsigned long long>(h_max, 4), 1024) + 1) & ~1ULL);
    const size_t fast_smem = HullFastLayout::bytes(fast_cap) * kHullWarps;
    int fast_grid = 1;
    Scratch<uint8_t> redo;
    if (n > 0) {
        GPL_TRY(redo.get(ctx, (size_t)n));
        GPL_CUDA(cudaFuncSetAttribute(k_hull_fast<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
        GPL_CUDA(cudaFuncSetAttribute(k_hull_fast<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
        int occ = 1;  // 5 CTAs per SM at 258 coordinates: 96 registers (a few spills; 128 registers / 4 CTAs measured the same)
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_hull_fast<true>, kHullWarps * 32, fast_smem) != cudaSuccess || occ < 1) occ = 1;
        (void)cudaGetLastError();
        fast_grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n, kHullWarps), (int64_t)kSMs * occ));
    }
    // pass: 0 = count only, 1 = write.  `off`/`dst` are the ring offsets and the output buffer of a writing pass.
    auto launch = [&](bool write, int64_t *cnt, const int64_t *off, double2 *dst) -> int {
        if (n == 0) return GPL_OK;
        if (write)
            k_hull_fast<true><<<fast_grid, kHullWarps * 32, fast_smem, ctx->stream>>>(in->type, n, xy, in->geom_off, in->part_off, in->ring_off, in->validity,
                                                                               fast_cap, cnt, off, dst, redo.p);
        else
            k_hull_fast<false><<<fast_grid, kHullWarps * 32, fast_smem, ctx->stream>>>(in->type, n, xy, in->geom_off, in->part_off, in->ring_off, in->validity,
                                                                                fast_cap, cnt, off, dst, redo.p);
        ctx->launches++;
        if (use_smem) {
            if (write) k_hull<true, true><<<grid, kHullWarps * 32, dyn, ctx->stream>>>(in->type, n, xy, in->geom_off, in->part_off, in->ring_off, in->validity, cap, workspace.p, cnt, off, dst, redo.p);
            else k_hull<false, true><<<grid, kHullWarps * 32, dyn, ctx->stream>>>(in->type, n, xy, in->geom_off, in->part_off, in->ring_off, in->validity, cap, workspace.p, cnt, off, dst, redo.p);
        } else {
            if (write) k_hull<true, false><<<grid, kHullWarps * 32, 0, ctx->stream>>>(in->type, n, xy, in->geom_off, in->part_off, in->ring_off, in->validity, cap, workspace.p, cnt, off, dst, redo.p);
            else k_hull<false, false><<<grid, kHullWarps * 32, 0, ctx->stream>>>(in->type, n, xy, in->geom_off, in->part_off, in->ring_off, in->validity, cap, workspace.p, cnt, off, dst, redo.p);
        }
        ctx->launches++;
        GPL_CUDA(cudaGetLastError());
        return GPL_OK;
    };
    Scratch<int64_t> ring_off, geom_off;
    GPL_TRY(ring_off.get(ctx, (size_t)n + 1));
    GPL_TRY(geom_off.get(ctx, (size_t)n + 1));
    Scratch<double> oxy;
    int64_t h_total = 0;
    // Single pass when a temporary of the upper-bound size fits (ring <= exterior coords + 2): the machine
    // runs once, writes each ring into its slot and the rings are compacted afterwards.  Otherwise two
    // passes (count, scan, re-run and write).
    const size_t ub_coords = (size_t)in->n_coords + 2 * (size_t)n + 2;
    // try to get the temporary from the context cache / the device; on OOM fall back to two passes
    Scratch<double> tmp;
    bool single = n > 0;
    if (single && tmp.get(ctx, ub_coords * 2) != GPL_OK) {
        single = false;
        (void)cudaGetLastError();
    }
    if (single) {
        Scratch<int64_t> ub, tmp_off;
        GPL_TRY(ub.get(ctx, (size_t)n + 1));
        GPL_TRY(tmp_off.get(ctx, (size_t)n + 1));
        GPL_LAUNCH(ctx, k_hull_upper, (int)ceil_div(n, 256), 256, 0, in->type, n, in->geom_off, in->part_off, in->ring_off, ub.p);
        GPL_TRY((exclusive_scan<int64_t, int64_t>(ctx, ub.p, n, tmp_off.p, nullptr)));
        GPL_TRY(launch(true, counts.p, tmp_off.p, reinterpret_cast<double2 *>(tmp.p)));
        GPL_TRY((exclusive_scan<int64_t, int64_t>(ctx, counts.p, n, ring_off.p, total.p)));
        GPL_CUDA(cudaMemcpyAsync(&h_total, total.p, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        GPL_CUDA(cudaStreamSynchronize(ctx->stream));
        GPL_TRY(oxy.get(ctx, (size_t)h_total * 2));
        const int cgrid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n, 8), (int64_t)kSMs * 8));
        GPL_LAUNCH(ctx, k_hull_compact, cgrid, 256, 0, n, reinterpret_cast<const double2 *>(tmp.p), tmp_off.p, ring_off.p,
                   reinterpret_cast<double2 *>(oxy.p));
        GPL_CUDA(cudaStreamSynchronize(ctx->stream));  // tmp returns to the cache when this scope ends
    } else {
        GPL_TRY(launch(false, counts.p, nullptr, nullptr));
        GPL_TRY((exclusive_scan<int64_t, int64_t>(ctx, counts.p, n, ring_off.p, total.p)));
        GPL_CUDA(cudaMemcpyAsync(&h_total, total.p, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        GPL_CUDA(cudaStreamSynchronize(ctx->stream));
        GPL_TRY(oxy.get(ctx, (size_t)h_total * 2));
        GPL_TRY(launch(true, nullptr, ring_off.p, reinterpret_cast<double2 *>(oxy.p)));
    }
    // geom_off = identity: geometry i owns ring i (a null input row becomes an empty, null polygon)
    GPL_LAUNCH(ctx, k_iota, (int)ceil_div(n + 1, 256), 256, 0, geom_off.p, n + 1);
    gpl_array *o = array_new(ctx, GPL_POLYGON);
    o->n_geoms = n, o->n_rings = n, o->n_coords = h_total;
    o->xy = oxy.take(), o->own_xy = true;
    o->ring_off = ring_off.take(), o->own_ring = true;
    o->geom_off = geom_off.take(), o->own_geom = true;
    o->validity = in->validity;  // shared with the input
    o->parent = const_cast<gpl_array *>(in);
    array_retain(o->parent);
    *out = o;
    return GPL_OK;
}
