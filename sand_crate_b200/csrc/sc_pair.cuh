// sc_pair.cuh - the two fused pair kernels of fp64 mode (density, force+integrate), and what they share with the
// mixed-precision kernels of sc_tile.cuh and the count kernel: the neighbor walk, the acceptance test, the force tail.
//
//   k_density  (K4)  collision_detector.py:52-121 pair discovery fused with crate.py:161-175 (populate_colliders),
//                    261-275 (pressure) and 337-342 (surface normals); emits one record per directed pair
//   k_force    (K5)  crate.py:343-353 tension, 309-310 gravity, 295-307 pressure, 316-323 viscosity,
//                    245-259 wall bounce, 177-200 continuous collision, 360-361 integration
//
// K4 walks, for the particle at sorted index s, the 3x3 cells around it and collects accepted neighbors in EXACTLY
// the reference's list order (SURVEY.md section 8(a) row N): same row ascending from s+1, next row ascending, same
// row descending from s-1, previous row descending, first 20 only.  Every neighbor quantity read is a
// start-of-tick snapshot (Jacobi), so there are no atomics on particle data.
#pragma once
#include "sc_common.cuh"

namespace sc {

template <typename Real> struct Vec2;
template <> struct Vec2<double> { typedef double2 type; };
template <> struct Vec2<float> { typedef float2 type; };

// pressure and surface normal of one particle, written by K4 as one vector store and gathered by K5 as one load
template <typename Real> struct PS;
template <> struct __align__(16) PS<float> { float p, sx, sy, pad_; };
template <> struct __align__(32) PS<double> { double p, sx, sy, pad_; };

// Per-thread neighbor list kept in shared memory, one column per thread (conflict-free: slot k of thread t is
// word k * SC_BLOCK + t).  An entry is the neighbor's sorted index in the low 28 bits and the relative cell
// (dr + 1) * 4 + (dc + 1) in the high 4.
#define SC_IDX_MASK 0x0FFFFFFFu
#define SC_K5_BATCH 2  // pairs whose loads K5 issues back to back (the pair loop is latency bound)
struct NbrList {
    uint32_t *col;
    __device__ __forceinline__ uint32_t get(int k) const { return col[k * SC_BLOCK]; }
    __device__ __forceinline__ void set(int k, uint32_t e) { col[k * SC_BLOCK] = e; }
};

// The reference's acceptance of a candidate pair, bit for bit: the x-window evaluated from the LOWER-sorted particle
// (collision_detector.py:106-119) and sqrt(dx*dx + dy*dy) <= d in fp64 (collision_detector.py:77-79).  Out of line:
// it only runs for candidates whose fp32 distance estimate falls inside a narrow band around d (see below).
static __device__ __noinline__ bool accept_exact(double2 ps, double2 pj, double d, int dr, bool fwd) {
    const double xlo = fwd ? ps.x : pj.x, xhi = fwd ? pj.x : ps.x;
    const double ylo = fwd ? ps.y : pj.y, yhi = fwd ? pj.y : ps.y;
    if (dr == 0) { if (!(xhi <= xlo + d)) return false; }
    else { if (!(xlo - d <= xhi && xhi <= xlo + d)) return false; }
    const double dx = xhi - xlo, dy = yhi - ylo;
    return sqrt(dx * dx + dy * dy) <= d;
}

// Phase 1 of K4.  Candidates are screened in fp32 on CELL-RELATIVE coordinates (`rel` = position minus the origin of
// the particle's own cell, |rel| < d, so an fp32 holds it to 6e-8 d): squared distance outside [1 - 4e-6, 1 + 4e-6]
// d^2 decides by itself (the fp32 evaluation error is below 1e-6 d^2, and a pair that close to or that far inside d
// passes / fails the reference's x-window as well); inside the band the reference's own fp64 arithmetic is replayed
// (accept_exact).  The decisions are therefore bit-identical to the reference's in both precision modes, and the
// bulk of the liquid never touches an fp64 instruction here.  Cell visiting order = reference list order:
//   forward : (0,0) beyond s, (0,+1), (+1,-1), (+1,0), (+1,+1)   ascending
//   backward: (0,0) before s, (0,-1), (-1,+1), (-1,0), (-1,-1)   descending            [(dr, dc), mirrored]
__device__ __forceinline__ int collect_neighbors(uint32_t s, uint32_t c, const Grid &g,
                                                 const uint32_t *cell_start,
                                                 const float2 *rel, const double2 *pos,
                                                 NbrList lst) {
    const float df = (float)g.d;
    const float hi = (df * df) * (1.0f + 4e-6f), lo = (df * df) * (1.0f - 4e-6f);
    const float2 rs = rel[s];
    // the 12 cell boundaries of the 3x3 block, loaded up front (independent loads)
    const uint32_t *cs0 = cell_start + c - 1, *csn = cs0 + g.ncols, *csp = cs0 - g.ncols;
    const uint32_t m0 = cs0[0], m1 = cs0[1], m2 = cs0[2], m3 = cs0[3];
    const uint32_t n0 = csn[0], n1 = csn[1], n2 = csn[2], n3 = csn[3];
    const uint32_t p0 = csp[0], p1 = csp[1], p2 = csp[2], p3 = csp[3];
    // four contiguous sorted ranges, each three cells wide (per-thread trip counts in a warp are alike even though
    // per-cell counts are not, so the warp stays converged):
    //   (s, m3) ascending, [n0, n3) ascending, [m0, s) descending, [p0, p3) descending
    int count = 0;
#define SC_SCAN_RANGE(FIRST, STOP, B1, B2, DR, ASC)                                                              \
    {                                                                                                            \
        const float by = rs.y - (float)(DR) * df;                                                                \
        /* count < 20 in the loop condition = trim_collisions, collision_detector.py:91-93 */                   \
        float2 rnext = rel[(FIRST) != (STOP) ? (FIRST) : s]; /* software pipelining: the load of candidate   */ \
        for (uint32_t j = (FIRST); j != (STOP) && count < SC_MAX_NEIGHBORS; j += (ASC) ? 1u : 0xFFFFFFFFu) {     \
            const float2 rj = rnext;                         /* j + 1 is in flight while j is being tested   */ \
            const uint32_t jn = j + ((ASC) ? 1u : 0xFFFFFFFFu);                                                  \
            rnext = rel[jn != (STOP) ? jn : s];                                                                  \
            /* x offset of the candidate's cell column relative to ours: (rel_j + (dc, dr) d) - rel_s */         \
            const float ox = (j >= (B2)) ? df : ((j >= (B1)) ? 0.0f : -df);                                      \
            const float dx = (rj.x + ox) - rs.x, dy = rj.y - by;                                                 \
            const float qd = fmaf(dx, dx, dy * dy);                                                              \
            /* qd > hi: surely farther than d (NaN lands here too: the reference rejects NaN); qd < lo: inside */ \
            if (qd <= hi && (qd < lo || accept_exact(pos[s], pos[j], g.d, (DR), (ASC)))) {                       \
                const int dc = (int)(j >= (B1)) + (int)(j >= (B2)) - 1;                                          \
                lst.set(count, j | ((uint32_t)(((DR) + 1) * 4 + (dc + 1)) << 28));                               \
                ++count;                                                                                         \
            }                                                                                                    \
        }                                                                                                        \
    }
    SC_SCAN_RANGE(s + 1, m3, m1, m2, 0, true)
    SC_SCAN_RANGE(n0, n3, n1, n2, 1, true)
    SC_SCAN_RANGE(s - 1, m0 - 1, m1, m2, 0, false)
    SC_SCAN_RANGE(p3 - 1, p0 - 1, p1, p2, -1, false)
#undef SC_SCAN_RANGE
    return count;
}

// crate.py:167-174 for one directed pair (i <- j): unit vector from the (noised) neighbor to i and the weight
// w = 1 - clip(dist / d, 0, 1) (crate.py:270).
struct PairGeom { double nx, ny, w; };

template <int kNoise>
__device__ __forceinline__ PairGeom pair_geom_f64(const DevParams &P, double2 pi, double2 pj, uint32_t uid_i,
                                                  uint32_t uid_j, const double *host_noise, uint32_t noise_index) {
    double qx = pj.x, qy = pj.y;
    if constexpr (kNoise != SC_NOISE_NONE) {
        double ux, uy;
        if constexpr (kNoise == SC_NOISE_HOST) {
            ux = host_noise[2 * (size_t)noise_index];
            uy = host_noise[2 * (size_t)noise_index + 1];
        } else {
            const uint32_t h = pair_noise_bits(P.tick_key, uid_i, uid_j);
            ux = (double)(h >> 16) * (1.0 / 65536.0);
            uy = (double)(h & 0xFFFFu) * (1.0 / 65536.0);
        }
        qx += (ux - 0.5) * P.d * P.level;
        qy += (uy - 0.5) * P.d * P.level;
    }
    const double rx = pi.x - qx, ry = pi.y - qy;
    const double dist = sqrt(rx * rx + ry * ry);
    PairGeom g;
    g.nx = rx / dist;
    g.ny = ry / dist;
    double cl = dist / P.d;
    if (cl < 0) cl = 0;
    if (cl > 1) cl = 1;
    g.w = 1 - cl;
    return g;
}

// crate.py:272 np.sum over a 1-D array: NumPy pairwise_sum (sequential below 8; 8 lanes + tail up to 20)
__device__ inline double np_sum_1d(const double *a, int n) {
    if (n < 8) {
        if (n == 0) return 0.0;
        double r = a[0];
        for (int i = 1; i < n; ++i) r += a[i];
        return r;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i = 8;
    if (n >= 16) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] += a[8 + j];
        i = 16;
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += a[i];
    return res;
}

// ------------------------------------------------------------------------------------------------------------
// K4: neighbor discovery, pair geometry, pressure p_i and surface normal s_i.
// One record per directed pair (i <- j) goes to the pair buffer (pair_j: neighbor index, pair_n: unit vector) and
// is consumed by K5, so the pair geometry - noise hash, reciprocal square root - is evaluated once per tick instead
// of twice.  HBM is the idle resource on this path (the kernels are issue / L1 bound), so 12 bytes per pair are a
// good trade.
template <int kNoise>  // kNoise: SC_NOISE_* resolved at compile time (no branch in the pair loop)
__global__ void __launch_bounds__(SC_BLOCK)
k_density(Counters *cnt, Grid g, DevParams P, const uint32_t *cell_start,
          const double2 *pos, const float2 *rel, const uint32_t *cell_key,
          const uint32_t *uid, const double *host_noise,
          const uint32_t *noise_off, const uint32_t *rank_of_uid,
          uint32_t *pair_j, double2 *pair_n,
          uint32_t *pair_off, uint8_t *pair_cnt, PS<double> *ps_out, NextWallClear next) {
    pdl_enter();
    clear_next_walls(next);
    __shared__ uint32_t s_list[SC_MAX_NEIGHBORS * SC_BLOCK];
    const uint32_t n = cell_start[g.ncells];
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = s < n;
    NbrList lst{s_list + threadIdx.x};
    int K = 0;
    if (live) K = collect_neighbors(s, cell_key[s], g, cell_start, rel, pos, lst);
    // the warp's records go to one contiguous chunk of the pair buffer (one atomic per warp, no block barrier: a
    // __syncthreads here made every warp wait for the block's slowest neighbor scan).  Where the chunk lands is
    // arbitrary, but it is only ever reached through pair_off, so results do not depend on it.
    const int lane = threadIdx.x & 31;
    uint32_t inc = (uint32_t)K;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
    uint32_t base = 0;
    if (lane == 31 && total) base = atomicAdd(&cnt->pair_cursor, total);
    base = __shfl_sync(0xffffffffu, base, 31);
    const uint32_t before = inc - (uint32_t)K;
    if (!live) return;
    const uint32_t off = base + before;
    pair_off[s] = off;
    pair_cnt[s] = (uint8_t)K;
    const uint32_t uid_s = uid[s];
    uint32_t nbase = 0u;
    if constexpr (kNoise == SC_NOISE_HOST) nbase = noise_off[rank_of_uid[uid_s]];
    double ax = 0, ay = 0;
    double wl[SC_MAX_NEIGHBORS];  // np.sum's pairwise order needs the list
    const double2 ps64 = pos[s];
    for (int k = 0; k < K; ++k) {
        const uint32_t j = lst.get(k) & SC_IDX_MASK;
        const PairGeom pg = pair_geom_f64<kNoise>(P, ps64, pos[j], uid_s, uid[j], host_noise, nbase + (uint32_t)k);
        pair_j[(size_t)off + k] = j;
        pair_n[(size_t)off + k] = make_double2(pg.nx, pg.ny);
        wl[k] = pg.w;
        const double c = (1 - pg.w) * pg.w;
        const double tx = c * pg.nx, ty = c * pg.ny;
        if (k == 0) { ax = tx; ay = ty; } else { ax += tx; ay += ty; }
    }
    double p = 0;
    if (K > 0) {
        const double pr = np_sum_1d(wl, K) - P.ignored;
        p = (pr > 0 || pr != pr) ? pr : 0.0;  // np.maximum(0, pr), crate.py:273
    }
    PS<double> o;
    o.p = p; o.sx = ax; o.sy = ay; o.pad_ = 0;
    ps_out[s] = o;
}

// NextKeys: K5 is the tick's last kernel and writes the new position of sorted particle s to pos_out[s]; the next tick's
// pre-pass would read that same array at that same index (the state is kept in the last tick's sorted order).  So K5 can
// run the next tick's key pass (key_particle) on the position it holds in registers, and the next tick goes straight to
// the cell scan.  `keys.cell_count == NULL`: not this tick (the host decides, see enqueue_forces).  What the pass writes
// belongs to the NEXT tick and none of it is read by K5: cell_key, wall_slot_cur and pos_cur are outputs only, and the
// wall bitmap, side list and its counter are the other tick parity's, which K4 cleared.
struct NextKeys { Grid g; KeyOut out; };

// Everything of K5 that follows the pair loop, for particle s: wall contact rows of F5, F3-F6 velocity updates, wall
// bounce, continuous collision, integration, and the next tick's key pass.  `visc(vx, vy, ax, ay)` supplies
// sum_j (v_j - v) (crate.py:319-323).
template <typename Real, bool kMonitor, typename ViscFn>
__device__ __forceinline__ void force_tail(uint32_t s, int K, Real p_i, Real tx, Real ty, Real qx, Real qy,
                                           const DevParams &P, const WallParams &W, const double2 ps,
                                           const typename Vec2<Real>::type v0, const bool touching,
                                           const uint32_t *wall_slot,
                                           const double2 *wall_pre, double2 *pos_out,
                                           typename Vec2<Real>::type *vel_out,
                                           double *monitor, const uint32_t *n_ptr,
                                           const NextKeys &nk, ViscFn visc) {
    typedef typename Vec2<Real>::type R2;
    auto store_pos = [&](double2 po) {
        pos_out[s] = po;
        if (nk.out.cell_count) key_particle<true>(nk.g, P, W, nk.out, s, po);
    };
    double mon[6] = {0, 0, 0, 0, 0, 0};
    double mpx = 0, mpy = 0;  // velocity before the current stage
    auto stage = [&](int q, double cx, double cy) {
        if constexpr (kMonitor) {
            const double ex = cx - mpx, ey = cy - mpy;
            mon[q] = sqrt(ex * ex + ey * ey);  // np.linalg.norm(velocity_diff, axis=1)
            mpx = cx; mpy = cy;
        }
    };
    // walls: contacts are recomputed from the position the particle had BEFORE apply_hard_wall_fix
    // (crate.py:216 runs before 202-211 and the vectors are never refreshed)
    int V = 0;
    double wnx = 0, wny = 0, wux = 0, wuy = 0;  // sequential sums for np.mean (crate.py:249-250)
    if (touching) {
        const double2 pre = wall_pre[wall_slot[s]];
        int nb[SC_MAX_BODIES];
        for (int b = 0; b < W.nbodies; ++b) nb[b] = 0;
        for (int q = 0; q < W.S; ++q) {
            double cx, cy;
            if (point_segment(pre.x, pre.y, W.seg[q][0], W.seg[q][1], W.seg[q][2], W.seg[q][3], cx, cy) <= P.touch)
                nb[W.seg_body[q]]++;
        }
        for (int q = 0; q < W.S; ++q) {
            double cx, cy;
            if (!(point_segment(pre.x, pre.y, W.seg[q][0], W.seg[q][1], W.seg[q][2], W.seg[q][3], cx, cy) <= P.touch))
                continue;
            const double vcx = (pre.x - cx) * 2, vcy = (pre.y - cy) * 2;  // crate.py:234, not normalised
            // W1b as written (crate.py:73-85): row V is overwritten by every body with more than V contacts
            double ux = 0, uy = 0;
            for (int b = 0; b < W.nbodies; ++b)
                if (nb[b] > V) {
                    const double rx = cx - W.kin[b][3], ry = cy - W.kin[b][4];
                    ux = W.kin[b][0] + ry * W.kin[b][2];
                    uy = W.kin[b][1] + (-rx) * W.kin[b][2];
                }
            // F5 virtual rows: n_k = vc_k, p_k = 0 (crate.py:286-293, 301-306)
            const Real ps_ = p_i + (Real)0;
            const Real fx = (Real)vcx * ps_, fy = (Real)vcy * ps_;
            if (K == 0 && V == 0) { qx = fx; qy = fy; } else { qx += fx; qy += fy; }
            if (V == 0) { wnx = vcx; wny = vcy; wux = ux; wuy = uy; }
            else { wnx += vcx; wny += vcy; wux += ux; wuy += uy; }
            ++V;
        }
    }

    const Real dt = sizeof(Real) == 4 ? (Real)P.f_dt : (Real)P.dt;
    Real vx = v0.x, vy = v0.y;
    if constexpr (kMonitor) { mpx = (double)vx; mpy = (double)vy; }
    if (K > 0) { vx += dt * tx; vy += dt * ty; }                       // F3, crate.py:352
    stage(0, (double)vx, (double)vy);
    if constexpr (sizeof(Real) == 4) { vx += P.f_dt_gx; vy += P.f_dt_gy; }
    else { vx += (Real)(P.dt * P.gx); vy += (Real)(P.dt * P.gy); }      // F4, crate.py:310
    stage(1, (double)vx, (double)vy);
    if (K + V > 0) {                                                     // F5, crate.py:297, 306
        const Real c = sizeof(Real) == 4 ? (Real)P.f_dt_amp : (Real)(P.dt * P.amp);
        vx += c * qx; vy += c * qy;
    }
    stage(2, (double)vx, (double)vy);
    {                                                                    // F6, crate.py:319-323
        Real ax = 0, ay = 0;
        visc(vx, vy, ax, ay);
        const Real c = sizeof(Real) == 4 ? (Real)P.f_dt_visc : (Real)(P.dt * P.visc);
        vx += c * ax; vy += c * ay;
    }
    stage(3, (double)vx, (double)vy);
    // Mixed precision, the bulk of the liquid (no wall contact, and the movement's box - taken in fp32, against a safe
    // rectangle shrunk by far more than fp32 rounding - stays clear of every padded segment): nothing of B1 / B2 applies,
    // and the fp64 detour below (conversions, products, min / max, compares: ~40 instructions) is skipped.  The result
    // is bit-identical to the general path's.
    bool bulk = false;
    if constexpr (sizeof(Real) == 4 && !kMonitor) {
        if (V == 0) {
            const float x0 = (float)ps.x, y0 = (float)ps.y;
            const float x1 = fmaf((float)vx, P.f_dt, x0), y1 = fmaf((float)vy, P.f_dt, y0);
            bulk = fminf(x0, x1) > W.safe_ccd_f32[0] && fmaxf(x0, x1) < W.safe_ccd_f32[1] &&
                   fminf(y0, y1) > W.safe_ccd_f32[2] && fmaxf(y0, y1) < W.safe_ccd_f32[3];
        }
    }
    if (bulk) {
        R2 vq;
        vq.x = vx; vq.y = vy;
        vel_out[s] = vq;
        store_pos(make_double2(ps.x + P.dt * (double)vq.x, ps.y + P.dt * (double)vq.y));      // I, crate.py:361
        return;
    }
    double dvx = (double)vx, dvy = (double)vy;
    if (V > 0) {                                                         // B1, crate.py:245-259
        const double Nx = wnx / (double)V, Ny = wny / (double)V;
        const double Ux = wux / (double)V, Uy = wuy / (double)V;
        const double nrm = sqrt(fma(Ny, Ny, Nx * Nx));                   // np.linalg.norm 1-D = sqrt(ddot)
        const double hx = Nx / nrm, hy = Ny / nrm;
        const double rvx = dvx - Ux, rvy = dvy - Uy;
        const double dot = fma(rvy, hy, rvx * hx);                       // np.dot = ddot
        if (dot < 0) {
            const double cx = -1 * dot * hx, cy = -1 * dot * hy;
            dvx += cx; dvy += cy;
            dvx += cx * P.decay; dvy += cy * P.decay;
        }
    }
    stage(4, dvx, dvy);
    {                                                                    // B2, crate.py:177-200
        const double mvx = dvx * P.dt, mvy = dvy * P.dt;
        const double bx = ps.x + mvx, by = ps.y + mvy;
        double f = 1.0;
        const double mxlo = fmin(ps.x, bx), mxhi = fmax(ps.x, bx), mylo = fmin(ps.y, by), myhi = fmax(ps.y, by);
        // one test for the bulk of the liquid: the movement stays inside a rectangle no padded segment reaches
        const bool clear = mxlo > W.safe_ccd[0] && mxhi < W.safe_ccd[1] && mylo > W.safe_ccd[2] && myhi < W.safe_ccd[3];
        if (!clear) {
            const double bax = bx - ps.x, bay = by - ps.y;
            for (int q = 0; q < 2 * W.S; ++q) {
                if (mxhi < W.pad_box[q][0] || mxlo > W.pad_box[q][1] || myhi < W.pad_box[q][2] || mylo > W.pad_box[q][3])
                    continue;  // the movement cannot reach this padded segment
                const double cx = W.pad[q][0], cy = W.pad[q][1], ex = W.pad[q][2], ey = W.pad[q][3];
                const double cdx = ex - cx, cdy = ey - cy;
                const bool opposite = (cdy * bax + (-cdx) * bay) < 0;    // geometry_utils.py:205
                if (!opposite) continue;
                const bool c1 = orientation(ps.x, ps.y, bx, by, cx, cy) != orientation(ps.x, ps.y, bx, by, ex, ey);
                const bool c2 = orientation(cx, cy, ex, ey, ps.x, ps.y) != orientation(cx, cy, ex, ey, bx, by);
                if (c1 && c2) {
                    const double acx = ps.x - cx, acy = ps.y - cy;
                    const double t = (acx * cdy - acy * cdx) / (cdx * mvy - cdy * mvx);  // geometry_utils.py:141-143
                    if (t < f) f = t;  // Python min(): NaN never wins (crate.py:199)
                }
            }
        }
        dvx *= f; dvy *= f;
    }
    stage(5, dvx, dvy);
    if constexpr (kMonitor) {
#pragma unroll
        for (int q = 0; q < 6; ++q) atomicAdd(&monitor[q], mon[q]);  // diagnostic mode only: speed is irrelevant
        if (threadIdx.x == 0 && blockIdx.x == 0) monitor[6] = (double)*n_ptr;
    }
    R2 vo;
    vo.x = (Real)dvx; vo.y = (Real)dvy;
    vel_out[s] = vo;
    double2 po;                                                          // I, crate.py:361
    po.x = ps.x + P.dt * (double)vo.x;
    po.y = ps.y + P.dt * (double)vo.y;
    store_pos(po);
}

// ------------------------------------------------------------------------------------------------------------
// K5: all forces, wall bounce, continuous collision and integration for particle s
// kMonitor: also accumulate, per force stage, the sum over particles of |dv| (the reference's ForceMonitor,
// utils/force_monitor.py:23-33, wraps exactly these six stages: crate.py:110-124)
// occupancy hint for K5 (forcing 5 or 6 blocks per SM spills the fp64 wall / crossing code: measured 2-8 us slower)
#ifndef SC_K5_MINBLOCKS
#define SC_K5_MINBLOCKS 1
#endif
template <bool kMonitor>
__global__ void __launch_bounds__(SC_BLOCK, SC_K5_MINBLOCKS)
k_force(const uint32_t *n_ptr, DevParams P, const __grid_constant__ WallParams W,
        const double2 *pos, const double2 *vel,
        const uint32_t *pair_j, const double2 *pair_n,
        const uint32_t *pair_off, const uint8_t *pair_cnt,
        const PS<double> *ps_in, const uint32_t *wall_bits,
        const uint32_t *wall_slot, const double2 *wall_pre,
        double2 *pos_out, double2 *vel_out,
        double *monitor, TickDuty duty, NextKeys nk) {
    pdl_enter();
    end_of_tick(duty, n_ptr);
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    const PS<double> me = ps_in[s];
    const double p_i = me.p;
    const uint32_t off = pair_off[s];
    const int K = pair_cnt[s];
    const double smooth = P.smooth, two_target = 2 * P.target;
    double tx = 0, ty = 0;  // F3 sum
    double qx = 0, qy = 0;  // F5 sum
    // batches of SC_K5_BATCH pairs: index loads, then the dependent gathers, then the arithmetic in list order - the loop is
    // latency bound (two dependent L2 round trips per pair), so the loads of a batch are issued back to back
    for (int k0 = 0; k0 < K; k0 += SC_K5_BATCH) {
        uint32_t jj[SC_K5_BATCH];
        double2 nn[SC_K5_BATCH];
        PS<double> pp[SC_K5_BATCH];
#pragma unroll
        for (int u = 0; u < SC_K5_BATCH; ++u)
            if (k0 + u < K) {
                jj[u] = pair_j[(size_t)off + k0 + u];
                nn[u] = pair_n[(size_t)off + k0 + u];
            }
#pragma unroll
        for (int u = 0; u < SC_K5_BATCH; ++u)
            if (k0 + u < K) pp[u] = ps_in[jj[u]];
#pragma unroll
        for (int u = 0; u < SC_K5_BATCH; ++u)
            if (k0 + u < K) {
                const double2 nv = nn[u];
                const PS<double> nb = pp[u];
                // F3 pass 2, crate.py:347-353
                const double ddx = me.sx - nb.sx, ddy = me.sy - nb.sy;
                const double align = (ddx * nv.x + ddy * nv.y) * smooth;
                const double fix = nb.p + p_i - two_target;
                const double cc = align + fix;
                const double ex = cc * nv.x, ey = cc * nv.y;
                // F5, crate.py:301-306
                const double ps_ = p_i + nb.p;
                const double fx = nv.x * ps_, fy = nv.y * ps_;
                if (k0 + u == 0) { tx = ex; ty = ey; qx = fx; qy = fy; }
                else { tx += ex; ty += ey; qx += fx; qy += fy; }
            }
    }

    // own position / velocity are only needed from here on: loading them late keeps the pair loop's register
    // footprint (and with it the occupancy that hides the gather latency of this untiled kernel) small
    const double2 ps_own = pos[s];
    const double2 v_own = vel[s];
    const bool touching = (wall_bits[s >> 5] >> (s & 31)) & 1u;
    force_tail<double, kMonitor>(s, K, p_i, tx, ty, qx, qy, P, W, ps_own, v_own, touching, wall_slot, wall_pre, pos_out,
                                 vel_out, monitor, n_ptr, nk, [&](double vx, double vy, double &ax, double &ay) {
        for (int q = 0; q < K; ++q) {
            const double2 vj = vel[pair_j[(size_t)off + q]];
            const double ex = vj.x - vx, ey = vj.y - vy;
            if (q == 0) { ax = ex; ay = ey; } else { ax += ex; ay += ey; }
        }
    });
}

}  // namespace sc
