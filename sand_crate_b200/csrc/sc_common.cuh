// sc_common.cuh - shared device-side definitions for the SandCrate particle step on sm_100a.
//
// Everything here restates ONE reference tick (David-Taub/sand_crate src/crate/crate.py:91-129) as per-particle
// device functions.  One translation unit (sc_api.cu), compiled with -fmad=false: NumPy never fuses multiply-add, so
// the fp64 parity kernels may not either; the fp32 production kernels spell out fmaf() where fusion is wanted.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/sandcrate.h"

#define SC_INVALID_CELL 0xFFFFFFFFu
#define SC_BLOCK 256
// particles per block of the tiled density kernel (sc_tile.cuh) = granularity of the window descriptors
#ifndef SC_TILE
#define SC_TILE 256
#endif

namespace sc {

// NO POINTER IN THIS LIBRARY IS DECLARED __restrict__.  With `const T *__restrict__` nvcc turns loads into
// ld.global.nc (LDG.E.CONSTANT), the non-coherent path, which is only defined for data that is read-only for the whole
// lifetime of the kernel.  Under programmatic dependent launch (below) a kernel's blocks are resident BEFORE the
// preceding kernel has finished writing that data, so non-coherent loads could (and, measured on B200, did) return
// stale lines: fp64 free runs were not reproducible from run to run and occasionally faulted, and went away with
// CUDA_LAUNCH_BLOCKING=1.  Plain loads are ordered by griddepcontrol.wait; they cost nothing measurable here.
//
// Programmatic dependent launch (sm_90+): the step's kernels are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so the next kernel's blocks may become resident while the
// current kernel drains.  pdl_enter() = let the dependent kernel start launching, then wait until everything the
// preceding kernel wrote is visible.  A no-op for kernels launched the ordinary way.
__device__ __forceinline__ void pdl_enter() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// uniform cell grid with cell edge = one particle diameter; row = floor(y / d) is the reference's strip index
// (collision_detector.py:126), col = floor(x / d) is ours (monotone in x, so a cell-major order
// (row, col, x, uid) is the same permutation as np.lexsort((x, row)), collision_detector.py:127).
struct Grid {
    double d;          // diameter
    double inv_d;      // 1 / d, only used to pre-screen floor(y / d) (see cell_of)
    int row_min;       // cell row index = row - row_min, clamped to [1, nrows - 2]
    int col_min;
    int nrows;
    int ncols;
    uint32_t ncells;
};

struct DevParams {
    double dt, r, d, touch;  // touch = r * 1.2 (crate.py:229)
    double decay, amp, ignored, level, visc, smooth, target, gx, gy;
    double box_lo, box_hi;   // -r, 1 + r  (crate.py:152)
    int noise_mode;
    uint64_t tick_key;
    // the fp32 kernels' constants, converted ONCE on the host (refresh_dev_params) with the same IEEE operations the
    // kernels used to spend on them per thread - an fp64 reciprocal and half a dozen fp64 -> fp32 conversions per
    // particle were ~5 % of the density kernel's instructions
    float f_d, f_inv_d, f_amp /* d * level */, f_band_hi, f_band_lo /* d^2 (1 +- 4e-6): the fp32 screen's certain zone */;
    float f_dt, f_dt_gx, f_dt_gy, f_dt_amp, f_dt_visc, f_smooth, f_two_target, f_ignored;
};

// ---- ensembles (DESIGN.md section 12): M members of one scene stepped as one particle set ----------------------------
// Member m's cells are m * ncells + its own cell of the scene's grid (whose margin rows and columns stay empty, so no 3x3
// neighborhood reaches another member), and its uids are (m << uid_bits) | local uid.  The ensemble instantiations of
// the step's kernels (kEns = true) take this as their LAST parameter, so the single-scene instantiations keep every
// parameter offset.  `params` holds each member's DevParams (noise_mode = its effective mode; tick_key unused: the key
// is tick_key(seed[m], tick), computed per thread from the launch's tick, so nothing is uploaded per tick).
struct Members {
    const DevParams *params;
    const unsigned long long *seed;
    const uint32_t *uid;  // the uids of the arrays the kernel indexes by particle
    unsigned long long tick;
    uint32_t uid_bits, ncells;  // identity bits of one member, cells of one member's grid
    int nrows;                  // rows of one member's grid
};

struct WallParams {
    int S;
    int nbodies;
    double seg[SC_MAX_SEGMENTS][4];       // ax, ay, bx, by                       (crate.py:69-71)
    double pad[2 * SC_MAX_SEGMENTS][4];   // pad_segments(segments, r)            (geometry_utils.py:146-172)
    int seg_body[SC_MAX_SEGMENTS];
    double kin[SC_MAX_BODIES][5];         // vcx, vcy, omega, posx, posy          (rigid_body.py:18-34)
    // conservative culls (never change a result, only skip work): a wall contact needs the particle inside the
    // segment's bounding box grown by the touch distance; a crossing needs the movement's box to meet the padded
    // segment's box.  (xmin, xmax, ymin, ymax), grown by a few ulps on the host.
    double seg_box[SC_MAX_SEGMENTS][4];
    double pad_box[2 * SC_MAX_SEGMENTS][4];
    // one rectangle (x0, x1, y0, y1; empty when x0 > x1) that no seg_box / no pad_box meets: the single test
    // that lets the bulk of the liquid skip the per-segment loops altogether
    double safe_contact[4];
    double safe_ccd[4];
    float safe_ccd_f32[4];  // safe_ccd shrunk by 1e-6: the mixed-precision kernel tests the movement in fp32 first
};

// ---- strip decomposition: what the wire looks like (kernels in sc_dist.cuh; the pre-pass reads it too) ----------------
#define SC_GHOST_BIT 0x80000000u
#define SC_WIRE_MIGRANT 0u
#define SC_WIRE_HALO 1u

// 16-byte header followed by `count` records
struct WireHeader { uint32_t count, overflow, too_far, pad_; };
struct __align__(8) WireRec { double px, py, vx, vy; uint32_t uid, kind; };  // 40 bytes

__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

struct UnpackSide { const WireHeader *hdr; const uint32_t *flag; };  // flag == NULL: the data is already there
// The strip unpack done by the PRE-PASS itself (sc_sort.cuh k_prepass): the blocks that cover the indices behind the
// particles this rank already holds wait for the neighbors' flags, read their records straight from the receive buffers,
// append them and go on with walls and cell keys for them - one launch less on the tick's critical path, and the wait for
// the neighbors hides behind the pass over the particles that were already here.
struct PrepassUnpack {
    int on;                 // 0: ordinary pass
    int vel_is_f64;
    UnpackSide lo, hi;
    uint32_t value, wire_cap;
    void *vel;              // float2* / double2*
    uint32_t *uid;
    WireHeader *send_lo, *send_hi;  // re-armed for the next pack
};


// device-resident counters, zeroed/updated on the stream (no host round trip in the step)
struct Counters {
    uint32_t n;          // live particles at the start of the tick (= after the previous tick's removal)
    uint32_t n_split;    // strips: the count before the neighbors' records were appended (k_dist_pack) = where the
                         // second, small wall / key pass of the tick starts (see enqueue_search)
    uint32_t n_wall[2];  // particles touching a wall, per tick parity (the force kernel of one tick may already fill
                         // the next tick's list while this tick's is being read, see NextKeys)
    uint32_t n_pairs;    // sum K_i (filled by the count kernel)
    uint32_t overflow;   // capacity problems seen on the device
    uint32_t pair_cursor;  // fp64 K4: next free record of the pair buffer (bump allocator, reset every tick)
    uint32_t n_tmp;        // scratch count (strip decomposition pack / readback)
    uint32_t n_untiled;    // blocks of the tiled K4 that ran in pass-through mode this tick (windows too large to stage)
};

// What the tick's LAST kernel (the force kernel) does for the NEXT tick, spread over its threads, so that a tick does
// not open with a clearing launch: zero the cell scan's tile descriptors and ticket and carry the live count (the scan
// total) into cnt->n.  The cell-count grid needs no clearing: k_place takes every count back to zero.
struct TickDuty {
    unsigned long long *scan_desc; uint32_t scan_words;
    Counters *cnt;
};
__device__ __forceinline__ void end_of_tick(const TickDuty &D, const uint32_t *n_ptr) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (uint32_t i = tid; i < D.scan_words; i += nth) D.scan_desc[i] = 0ull;
    if (tid == 0) D.cnt->n = *n_ptr;
}

// What the density kernel (K4) clears for the NEXT tick: the wall bitmaps and the wall side-list counter of the other
// tick parity.  Not the force kernel: when it computes the next tick's keys (NextKeys) it writes into exactly these.
struct NextWallClear {
    uint32_t *bits_a, *bits_b; uint32_t nbits;   // next tick's wall bitmaps (words)
    uint32_t *n_wall;                            // next tick's wall side-list counter
};
__device__ __forceinline__ void clear_next_walls(const NextWallClear &C) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (uint32_t i = tid; i < C.nbits; i += nth) { C.bits_a[i] = 0; C.bits_b[i] = 0; }
    if (tid == 0) *C.n_wall = 0;
}

// ---- counter-based pair noise (the production definition; oracle/step_oracle.c restates it) -------------
// Host side: tick_key = splitmix64 finalizer of (seed, tick).  Device side, per DIRECTED pair (i <- j), 32-bit
// arithmetic only: the two uids are spread with distinct odd multipliers, keyed with the two halves of tick_key
// folded together, and mixed with the lowbias32 finalizer (2 multiplies, 3 xor-shifts).  The high 16 bits of the
// result are the x uniform, the low 16 bits the y uniform (k / 65536: exact in fp32 and fp64 alike; the noise
// amplitude is 0.1 d, so the grain is 1.5e-6 d).  Bit 31 of a uid marks a ghost copy in the strip decomposition
// (sc_dist.cuh) and is not part of the identity.
__host__ __device__ inline uint64_t mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27; z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
__host__ __device__ inline uint64_t tick_key(uint64_t seed, uint64_t tick) {
    return mix64(seed * 0x9E3779B97F4A7C15ULL + tick);
}
__host__ __device__ inline uint32_t lowbias32(uint32_t x) {
    x ^= x >> 16; x *= 0x7FEB352Du;
    x ^= x >> 15; x *= 0x846CA68Bu;
    x ^= x >> 16;
    return x;
}
__host__ __device__ inline uint32_t pair_noise_bits(uint64_t tkey, uint32_t uid_i, uint32_t uid_j) {
    const uint32_t a = uid_i & 0x7FFFFFFFu, b = uid_j & 0x7FFFFFFFu;
    return lowbias32((a * 0x9E3779B1u) ^ (b * 0x85EBCA77u) ^ ((uint32_t)tkey ^ (uint32_t)(tkey >> 32)));
}
__device__ __forceinline__ uint32_t member_of(const Members &E, uint32_t uid) { return uid >> E.uid_bits; }
__device__ __forceinline__ DevParams member_params(const Members &E, uint32_t uid) {
    const uint32_t m = member_of(E, uid);
    DevParams p = E.params[m];
    p.tick_key = tick_key(E.seed[m], E.tick);
    return p;
}
// the kernel's own parameters, or the member's
template <bool kEns>
__device__ __forceinline__ const DevParams &pick_params(const DevParams &P, const DevParams &Pm) {
    if constexpr (kEns) return Pm;
    else return P;
}
// the uid the pair noise hashes: a member draws the noise of a separate context, so only its local identity counts
template <bool kEns>
__device__ __forceinline__ uint32_t noise_uid(const Members &E, uint32_t uid) {
    if constexpr (kEns) return uid & ((1u << E.uid_bits) - 1u);
    else return uid;
}

// ---- counter-based particle sources (production mode; oracle/step_oracle.c restates it) ---------------------
// Stream of source q at a tick: element j is u(j) = (mix64(source_key(tick_key, q) + (j + 1) * GOLDEN) >> 11) * 2^-53.
// j = 0 feeds the host's binomial draw of the emission count; particle k uses j = 1 + 4 k + {0: x, 1: y, 2: vx, 3: vy}.
__host__ __device__ inline uint64_t source_key(uint64_t tkey, uint32_t q) {
    return mix64(tkey ^ (0xD1B54A32D192ED03ULL * (uint64_t)(q + 1u)));
}
__host__ __device__ inline double source_uniform(uint64_t skey, uint64_t j) {
    return (double)(mix64(skey + (j + 1ull) * 0x9E3779B97F4A7C15ULL) >> 11) * (1.0 / 9007199254740992.0);
}

// the two uniforms as fp32 in [1, 2) (k / 65536 + 1): bits dropped straight into the mantissa, no int-to-float convert
__device__ __forceinline__ void pair_noise_f32_1to2(uint32_t h, float &fx, float &fy) {
    fx = __uint_as_float(0x3F800000u | ((h >> 9) & 0x007FFF80u));
    fy = __uint_as_float(0x3F800000u | ((h << 7) & 0x007FFF80u));
}

// ---- geometry_utils.py:7-39 for one (point, segment) -----------------------------------------------------
__device__ inline double point_segment(double px, double py, double ax, double ay, double bx, double by,
                                     double &cx, double &cy) {
    const double abx = bx - ax, aby = by - ay;
    const double apx = px - ax, apy = py - ay;
    const double rate = (apx * abx + apy * aby) / (abx * abx + aby * aby);
    double t = rate;  // np.clip(rate, 0, 1), NaN propagates
    if (t < 0) t = 0;
    if (t > 1) t = 1;
    cx = abx * t + ax;
    cy = aby * t + ay;
    const double dx = cx - px, dy = cy - py;
    return sqrt(dx * dx + dy * dy);
}

__device__ inline double sign_np(double v) {  // np.sign
    if (v > 0) return 1.0;
    if (v < 0) return -1.0;
    if (v == 0) return 0.0;
    return v;
}
__device__ inline double orientation(double px, double py, double qx, double qy, double rx, double ry) {
    return sign_np(((qy - py) * (rx - qx)) - ((qx - px) * (ry - qy)));  // geometry_utils.py:212-222
}

// floor(v / d) exactly as NumPy computes it (collision_detector.py:126), without paying for an fp64 division on
// every particle: v * (1/d) and v / d differ by at most a couple of ulps, so their floors can only differ when the
// product lands within that distance of an integer - only then is the true division evaluated.
static __device__ __noinline__ double floor_div_exact(double v, double d) { return floor(v / d); }
__device__ __forceinline__ double floor_div(double v, const Grid &g) {
    const double q = v * g.inv_d;
    const double f = floor(q);
    const double near = fmin(q - f, (f + 1.0) - q);
    if (!(near > fabs(q) * 1e-14)) return floor_div_exact(v, g.d);  // also NaN / inf
    return f;
}

// cell of a position; NaN / out-of-grid coordinates are clamped into the margin cells
__device__ inline uint32_t cell_of(const Grid &g, double x, double y, int &row_out) {
    const double fr = floor_div(y, g), fc = floor_div(x, g);
    int row = (fr >= -2.0e9 && fr <= 2.0e9) ? (int)fr : 0;
    int col = (fc >= -2.0e9 && fc <= 2.0e9) ? (int)fc : 0;
    row_out = row;
    int cr = row - g.row_min, cc = col - g.col_min;
    cr = cr < 1 ? 1 : (cr > g.nrows - 2 ? g.nrows - 2 : cr);
    cc = cc < 1 ? 1 : (cc > g.ncols - 2 ? g.ncols - 2 : cc);
    return (uint32_t)cr * (uint32_t)g.ncols + (uint32_t)cc;
}

// ------------------------------------------------------------------------------------------------------------
// K0 + K1 for ONE particle: the work of a tick's pre-pass, run either by k_prepass (sc_sort.cuh) or, for the next
// tick, by the previous tick's force kernel on the position it has just integrated (force_tail, sc_pair.cuh; see
// NextKeys).  One routine, so the two paths give the same bits.
//   kStep = true : remove_particles (crate.py:149-159), calc_virtual_colliders + apply_hard_wall_fix
//                  (crate.py:213-243, 202-211), then the cell key
//   kStep = false: cell key only (standalone detect_particle_collisions)
// Writes cell_key[i] (SC_INVALID_CELL for a removed particle), adds one to the particle's cell count (no value comes
// back: where a particle goes inside its cell is claimed later, by k_place), and for a particle the wall fix moves:
// its new position to pos[i], the old one to the wall side list, its slot there and its wall bit.
// INVARIANT: the particles counted here are exactly the particles k_place places - index below the clamped live count,
// key valid - because k_place takes each count back down to zero with one decrement per particle it places.  A count
// left above zero would shift every later cell of the next tick's scan.
struct KeyOut {
    uint32_t *cell_key, *cell_count;
    uint32_t *wall_bits, *wall_slot, *n_wall;
    double2 *pos, *wall_pre;
};
// kEns: the particle belongs to the ensemble member whose grid starts at cell `cell_base` (Members)
template <bool kStep, bool kEns = false>
__device__ __forceinline__ void key_particle(const Grid &g, const DevParams &P, const WallParams &W, const KeyOut &O,
                                             uint32_t i, double2 p, uint32_t cell_base = 0u) {
    if (kStep) {
        const bool out = (p.x < P.box_lo) | (p.x > P.box_hi) | (p.y < P.box_lo) | (p.y > P.box_hi);
        if (out) {
            O.cell_key[i] = SC_INVALID_CELL;
            return;
        }
        // one test for the bulk of the liquid: inside a rectangle that no segment's touch zone reaches
        const bool clear = p.x > W.safe_contact[0] && p.x < W.safe_contact[1] &&
                           p.y > W.safe_contact[2] && p.y < W.safe_contact[3];
        if (!clear) {
            int V = 0;
            double sx = 0, sy = 0;
            for (int q = 0; q < W.S; ++q) {
                if (p.x < W.seg_box[q][0] || p.x > W.seg_box[q][1] || p.y < W.seg_box[q][2] || p.y > W.seg_box[q][3])
                    continue;  // cannot be within the touch distance of this segment
                double cx, cy;
                const double dist = point_segment(p.x, p.y, W.seg[q][0], W.seg[q][1], W.seg[q][2], W.seg[q][3], cx, cy);
                if (dist <= P.touch) {
                    const double vcx = (p.x - cx) * 2, vcy = (p.y - cy) * 2;  // crate.py:234
                    double rel = P.r / sqrt(vcx * vcx + vcy * vcy);          // crate.py:206
                    if (rel < 0.5) rel = 0.5;
                    const double ex = vcx * (rel - 0.5), ey = vcy * (rel - 0.5);
                    if (V == 0) { sx = ex; sy = ey; } else { sx += ex; sy += ey; }
                    ++V;
                }
            }
            if (V > 0) {
                const uint32_t ws = atomicAdd(O.n_wall, 1u);
                O.wall_pre[ws] = p;  // contacts are re-derived from this position by the force kernel
                O.wall_slot[i] = ws;
                atomicOr(&O.wall_bits[i >> 5], 1u << (i & 31));
                p.x += sx;
                p.y += sy;
                O.pos[i] = p;
            }
        }
    }
    int row;
    uint32_t c = cell_of(g, p.x, p.y, row);
    if constexpr (kEns) c += cell_base;
    atomicAdd(&O.cell_count[c], 1u);  // result unused: a fire-and-forget reduction (RED), no round trip
    O.cell_key[i] = c;
}

// total order used inside a cell: x ascending (NaN last, like np.lexsort), ties by uid (lexsort is stable and
// original index order == uid order)
__device__ inline bool x_less(double a, double b) { return a < b || (b != b && a == a); }

// exclusive prefix sum over the NT threads of a block; `total` = sum over the block
template <int NT>
__device__ inline uint32_t block_exclusive_scan_n(uint32_t v, uint32_t &total) {
    __shared__ uint32_t warp_sums[NT / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = lane < NT / 32 ? warp_sums[lane] : 0;
#pragma unroll
        for (int o = 1; o < NT / 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        if (lane < NT / 32) warp_sums[lane] = w;
    }
    __syncthreads();
    const uint32_t base = wid ? warp_sums[wid - 1] : 0;
    total = warp_sums[NT / 32 - 1];
    __syncthreads();
    return base + inc - v;
}
__device__ inline uint32_t block_exclusive_scan(uint32_t v, uint32_t &total) {
    return block_exclusive_scan_n<SC_BLOCK>(v, total);
}

}  // namespace sc
