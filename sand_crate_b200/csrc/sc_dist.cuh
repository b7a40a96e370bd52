// sc_dist.cuh - strip decomposition across GPUs: the pack kernel of the per-tick boundary exchange (the unpack is done
// by the step's pre-pass, k_prepass<..., true> in sc_sort.cuh), the owned-particle readback and the re-cut histogram.
//
// The reference's own neighbor search is a 1-D strip decomposition in y with strip height one diameter
// (collision_detector.py:10-31, 124-128); the same rows are the multi-GPU partition unit.  Rank k owns the cell rows
// [row_lo, row_hi).  Every tick, BEFORE the step:
//   pack    drops last tick's ghosts, keeps particles whose row is still owned, turns particles whose row left the
//           strip into MIGRANT records for the neighbor (and keeps them here as ghosts for this tick), and copies
//           owned particles within `halo` rows of a cut into HALO records for that neighbor
//   (host)  exchanges the two fixed-capacity buffers with rank-1 / rank+1 (NCCL send/recv over NVLink)
//   unpack  appends received migrants as owned particles and received halos as ghosts
// and the ordinary single-GPU step then runs on owned + ghosts.  A ghost is a full particle (it is sorted, gets
// its own pressure and normal, is integrated) whose results are simply discarded by the next pack; with a halo of
// 4 rows every owned particle sees exactly the neighbors, pressures and normals it would see in the global
// computation, in the same order, so fp64 results are bit-identical to a single-GPU run (DESIGN.md section 6).
#pragma once
#include "sc_sort.cuh"

namespace sc {

struct DistCfg {
    long long row_lo, row_hi;  // owned rows: row_lo <= floor(y / d) < row_hi
    long long far_lo, far_hi;  // rows owned by the two neighbors: far_lo <= row < row_lo below, row_hi <= row < far_hi
                               // above.  A migrant must land INSIDE its neighbor's strip (anything further would need a
                               // second hop: the too_far flag); by default the reach is one halo.
    int halo;                  // rows
    int has_lo, has_hi;        // neighbors exist
    int reach_set;             // far_lo / far_hi were given by the caller
    uint32_t cap;              // records per wire buffer
};

// One atomic per WARP on the buffer's record counter, not one per record: the lanes that have a record for this buffer
// are counted with a ballot, the first of them reserves the run, every lane takes its place in it.  (One atomic per
// record meant ~12 000 serialized operations on a single address per tick and side: ~6 us of L2 atomic unit time.)
// Must be called by all 32 lanes.
__device__ __forceinline__ uint32_t wire_reserve(bool want, uint32_t *counter) {
    const uint32_t mask = __ballot_sync(0xffffffffu, want);
    if (!mask) return 0u;
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    uint32_t base = 0u;
    if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + (uint32_t)__popc(mask & ((1u << lane) - 1u));
}
__device__ __forceinline__ void wire_store(WireHeader *h, WireRec *recs, uint32_t cap, uint32_t k, double2 p, double vx,
                                           double vy, uint32_t uid, uint32_t kind) {
    if (k >= cap) { h->overflow = 1u; return; }
    WireRec r;
    r.px = p.x; r.py = p.y; r.vx = vx; r.vy = vy; r.uid = uid; r.kind = kind;
    recs[k] = r;
}

// A pass over the particle arrays, in place (no compaction: the arrays keep the previous tick's sorted order, which is
// what makes the next tick's gathers nearly coalesced):
//   last tick's ghost      -> killed: its x becomes +inf, so this tick's remove_particles pass (k_prepass) drops it
//   row left the strip     -> MIGRANT record for the neighbor; stays here, re-tagged as a ghost, for this tick
//   owned, near a cut      -> HALO record(s)
// n_in_ptr = live count left by the previous tick (its scan total) or cnt->n; it is copied to cnt->n and cnt->n_split,
// behind which the step's pre-pass appends what the neighbors send.  The send headers' counts are zero on entry (the
// pre-pass re-arms them once the previous tick's buffers have left).
//
// Only the rows near a cut can hold any of the three.  The arrays are in the last tick's sorted order (cell rows
// ascending), so those rows are two index ranges, [0, A) and [B, n), read off the last tick's cell boundaries
// (PackRange): the kernel then touches a few percent of the particles instead of all of them.  Without a valid search
// state (first tick, after a re-grid) the pass covers everything.
//
// kDirect (the NVLink transport): the records are written straight into the neighbor's receive buffer through a
// peer-mapped pointer - pack and transfer are ONE kernel, the bytes cross NVLink as they are produced - and the last
// block to finish publishes the record count and raises the neighbor's flag (release, system scope); the neighbor's
// pre-pass, running on its own GPU, acquires it.
struct PackRange {
    const uint32_t *cell_start;  // last tick's cell boundaries, or NULL: cover all particles
    uint32_t cell_a, cell_b;     // first cell of the first row above the lower boundary zone / of the upper boundary zone
};
struct PackOut {
    WireHeader *hdr;   // LOCAL header: record counter (atomic), sticky overflow / too_far marks
    WireRec *recs;     // where the records go: the local send buffer, or the neighbor's receive buffer (kDirect)
    WireHeader *peer_hdr; uint32_t *peer_flag;  // kDirect only
};

template <typename Real, bool kDirect>
__global__ void __launch_bounds__(SC_BLOCK)
k_dist_pack(Counters *cnt, const uint32_t *n_in_ptr, Grid g, DistCfg D, PackRange R,
            double2 *pos, const typename Vec2<Real>::type *vel,
            uint32_t *uid, PackOut lo, PackOut hi, uint32_t *done, uint32_t value) {
    pdl_enter();
    const uint32_t n_in = *n_in_ptr;
    if (blockIdx.x == 0 && threadIdx.x == 0) { cnt->n = n_in; cnt->n_split = n_in; }
    // the work list: [0, A) and [B, n_in) in zone mode, [0, n_in) otherwise; a FEW fat blocks walk it with a grid
    // stride (every block ends with a system-scope fence in the direct mode: 1 500 thin blocks spent more time in
    // fences than in packing)
    uint32_t A = n_in, B = n_in;
    if (R.cell_start) {
        A = D.has_lo ? R.cell_start[R.cell_a] : 0u;
        B = D.has_hi ? R.cell_start[R.cell_b] : n_in;
        if (B > n_in) B = n_in;
        if (A > B) A = B;
    }
    const uint32_t total = A + (n_in - B);
    for (uint32_t base = blockIdx.x * blockDim.x; base < total; base += gridDim.x * blockDim.x) {
    const uint32_t idx = base + threadIdx.x;
    const uint32_t i = idx < A ? idx : (idx < total ? B + (idx - A) : n_in);
    // decide (divergent), then reserve and write (warp-uniform control flow: wire_reserve needs all lanes)
    int kind_lo = -1, kind_hi = -1;  // record kind for the lower / upper neighbor, -1 = none
    uint32_t u = 0u;
    double2 p = make_double2(0, 0);
    if (i < n_in) {
        u = uid[i];
        if (u & SC_GHOST_BIT) {  // its owner has the authoritative copy
            pos[i].x = __longlong_as_double(0x7FF0000000000000LL);
        } else {
            p = pos[i];
            const double fr = floor_div(p.y, g);
            const long long row = (fr >= -9.0e18 && fr <= 9.0e18) ? (long long)fr : 0;  // NaN: stays where it is
            const bool below = row < D.row_lo && D.has_lo, above = row >= D.row_hi && D.has_hi;
            if (below) {
                if (row < D.far_lo) lo.hdr->too_far = 1u;
                kind_lo = (int)SC_WIRE_MIGRANT;
            } else if (above) {
                if (row >= D.far_hi) hi.hdr->too_far = 1u;
                kind_hi = (int)SC_WIRE_MIGRANT;
            } else {
                if (D.has_lo && row < D.row_lo + D.halo) kind_lo = (int)SC_WIRE_HALO;
                if (D.has_hi && row >= D.row_hi - D.halo) kind_hi = (int)SC_WIRE_HALO;
            }
            if (below || above) uid[i] = u | SC_GHOST_BIT;
        }
    }
    const uint32_t k_lo = wire_reserve(kind_lo >= 0, &lo.hdr->count), k_hi = wire_reserve(kind_hi >= 0, &hi.hdr->count);
    if (kind_lo >= 0 || kind_hi >= 0) {
        const typename Vec2<Real>::type v = vel[i];
        if (kind_lo >= 0) wire_store(lo.hdr, lo.recs, D.cap, k_lo, p, (double)v.x, (double)v.y, u, (uint32_t)kind_lo);
        if (kind_hi >= 0) wire_store(hi.hdr, hi.recs, D.cap, k_hi, p, (double)v.x, (double)v.y, u, (uint32_t)kind_hi);
    }
    }
    if constexpr (kDirect) {
        __threadfence_system();  // this block's records have reached the neighbor before it is counted as done
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t prev = atomicAdd(done, 1u);
            if (prev == gridDim.x - 1) {  // every block's records are out: publish the counts, raise the flags
                *done = 0u;
                __threadfence();
                if (D.has_lo) {
                    const uint32_t c = *(volatile uint32_t *)&lo.hdr->count;
                    lo.peer_hdr->count = c < D.cap ? c : D.cap;
                    st_release_sys(lo.peer_flag, value);
                }
                if (D.has_hi) {
                    const uint32_t c = *(volatile uint32_t *)&hi.hdr->count;
                    hi.peer_hdr->count = c < D.cap ? c : D.cap;
                    st_release_sys(hi.peer_flag, value);
                }
            }
        }
    }
}

// owned particles (no ghosts) compacted into staging arrays for readback; order is arbitrary, uids identify rows
template <typename Real>
__global__ void __launch_bounds__(SC_BLOCK)
k_dist_collect_owned(const uint32_t *n_ptr, const double2 *pos,
                     const typename Vec2<Real>::type *vel, const uint32_t *uid,
                     double2 *pos_out, double2 *vel_out, uint32_t *uid_out,
                     uint32_t *n_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *n_ptr) return;
    const uint32_t u = uid[i];
    if (u & SC_GHOST_BIT) return;
    const uint32_t k = atomicAdd(n_out, 1u);
    pos_out[k] = pos[i];
    const typename Vec2<Real>::type v = vel[i];
    vel_out[k] = make_double2((double)v.x, (double)v.y);
    uid_out[k] = u;
}

// per-row WORK of the owned particles (input of the partition re-cut): hist[row - row0], rows outside are clamped.
// A particle weighs work_base + K_i, K_i = its directed pairs of the last tick: the pair kernels are two thirds of a tick,
// their cost grows with K, and K is anything but uniform - the bottom strip of the settled 64M column holds 10.5 pairs
// per particle, the top 4.4 - so strips of equal particle COUNT are not strips of equal time.  work_base = 2 is
// calibrated on the 64M dam break cut in two (profiles/r3_work_model_2gpu.txt: 13 -> 3.608 ms per tick, 5 -> 3.529,
// 2 -> 3.456, 0 -> 3.516; the single-GPU tick halved would be 3.27): the pair-independent work (sort, staging) weighs
// like two pairs, because a dense region also costs more candidates to screen per particle.  A quadratic term in K
// over-corrects (3.73 / 3.97 ms).  Without a pair count (no tick yet) every particle weighs the same.
// The arrays are in the last tick's cell-major order, so a block's 256 particles lie in a handful of adjacent rows: the
// block sums them in shared memory (a window of SC_HIST_WIN rows above its lowest one; a warp wholly in one row adds one
// summed value) and issues one global atomic per row it touched - instead of one per particle, 32M of them on a few
// dozen hot addresses in the 64M scene (8 ms; profiles/r3f_*).  Rows outside the window fall back to global atomics.
#define SC_HIST_WIN 64
__global__ void __launch_bounds__(SC_BLOCK)
k_dist_row_hist(const uint32_t *n_ptr, Grid g, const double2 *pos,
                const uint32_t *uid, const uint8_t *pair_cnt, long long row0, int nrows, unsigned long long *hist,
                uint32_t work_base) {
    __shared__ int s_min;
    __shared__ uint32_t s_h[SC_HIST_WIN];
    if (threadIdx.x == 0) s_min = 0x7fffffff;
    if (threadIdx.x < SC_HIST_WIN) s_h[threadIdx.x] = 0u;
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < *n_ptr && !(uid[i] & SC_GHOST_BIT);
    int bin = 0x7fffffff;
    uint32_t w = 0;
    if (live) {
        const double fr = floor_div(pos[i].y, g);
        long long row = (fr >= -9.0e18 && fr <= 9.0e18) ? (long long)fr : row0;
        row = row < row0 ? row0 : (row >= row0 + nrows ? row0 + nrows - 1 : row);
        bin = (int)(row - row0);
        w = work_base + (pair_cnt ? pair_cnt[i] : 0u);
    }
    const int wmin = __reduce_min_sync(0xffffffffu, bin);
    if ((threadIdx.x & 31) == 0 && wmin != 0x7fffffff) atomicMin(&s_min, wmin);
    __syncthreads();
    const int base = s_min;
    const bool uniform = __all_sync(0xffffffffu, bin == wmin);   // dead lanes (bin = INT_MAX) make a warp non-uniform
    if (uniform) {
        const uint32_t sum = __reduce_add_sync(0xffffffffu, w);
        if ((threadIdx.x & 31) == 0 && live) {
            if (bin - base < SC_HIST_WIN) atomicAdd(&s_h[bin - base], sum);
            else atomicAdd(&hist[bin], (unsigned long long)sum);
        }
    } else if (live) {
        if (bin - base < SC_HIST_WIN) atomicAdd(&s_h[bin - base], w);
        else atomicAdd(&hist[bin], (unsigned long long)w);
    }
    __syncthreads();
    if (threadIdx.x < SC_HIST_WIN && s_h[threadIdx.x]) atomicAdd(&hist[base + threadIdx.x], (unsigned long long)s_h[threadIdx.x]);
}

__global__ void k_wire_reset(WireHeader *a, WireHeader *b) {
    a->count = 0; a->overflow = 0; a->too_far = 0; a->pad_ = 0;
    b->count = 0; b->overflow = 0; b->too_far = 0; b->pad_ = 0;
}

}  // namespace sc
