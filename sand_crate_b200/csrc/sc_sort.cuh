// sc_sort.cuh - precision-independent kernels of the step: wall pre-pass + cell keys (K0/K1), exclusive scan,
// counting-sort placement, in-cell rank + gather (K2/K3), neighbor count/list taps and the uid -> rank map.
// All position arithmetic here is fp64 without FMA contraction, so cell keys, sorted order and neighbor lists
// are bit-identical to the reference's in BOTH precision modes.
#pragma once
#include "sc_pair.cuh"
#include "sc_tile.cuh"

namespace sc {

// ------------------------------------------------------------------------------------------------------------
// K0 + K1 (key_particle, sc_common.cuh) as a launch of its own.  One thread per particle in the order the previous tick
// left them (that order is the previous tick's sorted order, so neighbouring threads touch neighbouring cells).  Runs
// when the previous tick's force kernel did not already do this work (NextKeys): the first tick, a tick after the host
// changed the state, the walls or the parameters, and every tick of a strip.
// particles per thread: the kernel is a chain of long-latency operations (position load, then the stores), so
// independent chains are interleaved (4 measured the same as 2)
#ifndef SC_PREPASS_ILP
#define SC_PREPASS_ILP 2
#endif
// kEns: an ensemble (Members, sc_common.cuh); `g` is then the grid of ONE member
template <bool kStep, bool kUnpack = false, bool kEns = false>  // kUnpack: the strip variant that appends the neighbors' records itself
__global__ void __launch_bounds__(SC_BLOCK, 6)  // the wall path may spill; it is rare
k_prepass(Counters *cnt, Grid g, DevParams P, const __grid_constant__ WallParams W, KeyOut O, uint32_t cap,
          PrepassUnpack U, Members E) {
    pdl_enter();
    const uint32_t b0 = blockIdx.x * (SC_BLOCK * SC_PREPASS_ILP);
    const uint32_t i0 = b0 + threadIdx.x;
    // the positions are requested BEFORE the live count is known (any index below the capacity is readable): the count
    // is itself a device-resident value, and waiting for it first put one more memory latency at the head of every thread
    double2 p[SC_PREPASS_ILP];
#pragma unroll
    for (int u = 0; u < SC_PREPASS_ILP; ++u) {
        const uint32_t i = i0 + u * SC_BLOCK;
        if (i < cap) p[u] = O.pos[i];
    }
    // every kernel bounds its indices by the count, so the count itself must never exceed the arrays
    uint32_t n = cnt->n < cap ? cnt->n : cap;
    if (blockIdx.x == 0 && threadIdx.x == 0 && cnt->n > cap) cnt->overflow = 1u;
    // strips: the neighbors' records are appended HERE (PrepassUnpack).  n_own = the particles already held; a record's
    // place is a pure function of its position in its buffer (lower neighbor's first), so the order is deterministic.
    uint32_t n_own = n, c_lo = 0u;
    if constexpr (kUnpack) {
        __shared__ uint32_t s_cnt[2];
        n_own = cnt->n_split < cap ? cnt->n_split : cap;
        n = n_own;
        if (b0 >= n_own + 2u * U.wire_cap) return;  // behind anything the neighbors can send
        if (b0 + SC_BLOCK * SC_PREPASS_ILP > n_own) {  // this block reaches into the appended range: it needs the records
            if (threadIdx.x == 0) {
                if (U.lo.hdr && U.lo.flag) while ((int)(ld_acquire_sys(U.lo.flag) - U.value) < 0) __nanosleep(64);
                if (U.hi.hdr && U.hi.flag) while ((int)(ld_acquire_sys(U.hi.flag) - U.value) < 0) __nanosleep(64);
                const uint32_t a = U.lo.hdr ? (U.lo.hdr->count < U.wire_cap ? U.lo.hdr->count : U.wire_cap) : 0u;
                const uint32_t b = U.hi.hdr ? (U.hi.hdr->count < U.wire_cap ? U.hi.hdr->count : U.wire_cap) : 0u;
                s_cnt[0] = a; s_cnt[1] = b;
                if (b0 <= n_own) {  // the one block that holds index n_own publishes the new count, re-arms the send buffers
                    cnt->n = n_own + a + b;   // (the next kernels clamp it and raise the flag)
                    if (n_own + a + b > cap) cnt->overflow = 1u;
                    U.send_lo->count = 0u; U.send_hi->count = 0u;
                }
            }
            __syncthreads();
            c_lo = s_cnt[0];
            const uint32_t total = n_own + c_lo + s_cnt[1];
            n = total < cap ? total : cap;
#pragma unroll
            for (int u = 0; u < SC_PREPASS_ILP; ++u) {
                const uint32_t i = i0 + u * SC_BLOCK;
                if (i < n_own || i >= n) continue;
                const uint32_t k = i - n_own;
                const WireRec r = k < c_lo ? reinterpret_cast<const WireRec *>(U.lo.hdr + 1)[k]
                                           : reinterpret_cast<const WireRec *>(U.hi.hdr + 1)[k - c_lo];
                p[u] = make_double2(r.px, r.py);
                O.pos[i] = p[u];
                if (U.vel_is_f64) reinterpret_cast<double2 *>(U.vel)[i] = make_double2(r.vx, r.vy);
                else reinterpret_cast<float2 *>(U.vel)[i] = make_float2((float)r.vx, (float)r.vy);
                U.uid[i] = r.kind == SC_WIRE_HALO ? (r.uid | SC_GHOST_BIT) : r.uid;
            }
        }
    }
#pragma unroll
    for (int u = 0; u < SC_PREPASS_ILP; ++u) {
        const uint32_t i = i0 + u * SC_BLOCK;
        if constexpr (kEns) {
            if (i < n) key_particle<kStep, true>(g, P, W, O, i, p[u], member_of(E, E.uid[i]) * E.ncells);
        } else {
            if (i < n) key_particle<kStep>(g, P, W, O, i, p[u]);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// exclusive scan of a u32 array, out of place (in == out is allowed), total written to out[n].
// 16 items per thread as four 128-bit accesses: a warp request covers 2 KB contiguous.
#define SC_SCAN_ITEMS 16
// few, large tiles (256- and 512-thread tiles measured 2-4 us slower on the 1.8M-cell grid; a row-wise scan without
// any look-back - one block per cell row, row totals accumulated by the pre-pass - measured 6 us slower in the scan
// and 6 us slower in the pre-pass)
#ifndef SC_SCAN_THREADS
#define SC_SCAN_THREADS 1024
#endif
#define SC_SCAN_TILE (SC_SCAN_THREADS * SC_SCAN_ITEMS)

__device__ __forceinline__ void scan_load(const uint32_t *a, uint32_t n, uint32_t base, uint32_t (&item)[SC_SCAN_ITEMS]) {
    if (base + SC_SCAN_ITEMS <= n) {
        const uint4 *p = reinterpret_cast<const uint4 *>(a + base);  // base is a multiple of 16 items
#pragma unroll
        for (int q = 0; q < SC_SCAN_ITEMS / 4; ++q) {
            const uint4 v = p[q];
            item[4 * q] = v.x; item[4 * q + 1] = v.y; item[4 * q + 2] = v.z; item[4 * q + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int q = 0; q < SC_SCAN_ITEMS; ++q) item[q] = (base + q < n) ? a[base + q] : 0u;
    }
}

// Single-pass exclusive scan: one launch, 8 bytes of traffic per item.  Tiles take their index from a ticket counter,
// so a tile's predecessors are always resident or done and waiting on them cannot deadlock.
// Tile descriptor = (status << 32) | value, written / read as one 64-bit word: status 1 = tile aggregate published.  `desc` (one word per tile) and `ticket` must be zero at launch.
__device__ __forceinline__ unsigned long long ld_desc(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_desc(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(SC_SCAN_THREADS)
k_scan_lookback(const uint32_t *in, uint32_t *out, uint32_t n, unsigned long long *desc,
                uint32_t *ticket) {
    pdl_enter();
    __shared__ uint32_t s_tile, s_prefix;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint32_t base = tile * SC_SCAN_TILE + threadIdx.x * SC_SCAN_ITEMS;
    uint32_t item[SC_SCAN_ITEMS];
    scan_load(in, n, base, item);
    uint32_t v = 0;
#pragma unroll
    for (int q = 0; q < SC_SCAN_ITEMS; ++q) v += item[q];
    uint32_t total;
    const uint32_t before = block_exclusive_scan_n<SC_SCAN_THREADS>(v, total);
    // publish this tile's aggregate, then read ALL predecessors' aggregates in parallel (one L2 round trip instead
    // of a serial chain of look-back windows: with every tile starting at once, tile k would otherwise walk k / 32
    // windows).  Lower tickets are always resident or finished, so the spin cannot deadlock.
    if (threadIdx.x == 0) st_desc(desc + tile, (1ull << 32) | total);
    uint32_t part = 0;
    for (uint32_t t = threadIdx.x; t < tile; t += SC_SCAN_THREADS) {
        unsigned long long d;
        do { d = ld_desc(desc + t); } while ((d >> 32) == 0ull);
        part += (uint32_t)d;
    }
    uint32_t prefix;
    block_exclusive_scan_n<SC_SCAN_THREADS>(part, prefix);
    if (threadIdx.x == 0) s_prefix = prefix;
    __syncthreads();
    uint32_t run = s_prefix + before;
#pragma unroll
    for (int q = 0; q < SC_SCAN_ITEMS; ++q) {
        const uint32_t t = item[q];
        item[q] = run;
        run += t;
    }
    if (base + SC_SCAN_ITEMS <= n) {
        uint4 *p = reinterpret_cast<uint4 *>(out + base);
#pragma unroll
        for (int q = 0; q < SC_SCAN_ITEMS / 4; ++q) p[q] = make_uint4(item[4 * q], item[4 * q + 1], item[4 * q + 2], item[4 * q + 3]);
    } else {
#pragma unroll
        for (int q = 0; q < SC_SCAN_ITEMS; ++q)
            if (base + q < n) out[base + q] = item[q];
    }
    if (tile == gridDim.x - 1 && threadIdx.x == SC_SCAN_THREADS - 1) out[n] = run;  // grand total
}

// ------------------------------------------------------------------------------------------------------------
// K2: counting-sort placement.  A particle claims its place inside its cell by taking one off the cell's count
// (key_particle counted it): the returned value minus one is a slot in [0, count), and after the last claim every
// count is zero again - the grid is ready for the next tick's key pass without a clearing pass.  The order inside a
// cell is arbitrary here; k_rank_gather makes it deterministic.
#define SC_PLACE_ILP 4
__global__ void __launch_bounds__(SC_BLOCK)
k_place(const Counters *cnt, const uint32_t *cell_key, uint32_t *cell_count,
        const uint32_t *cell_start, uint32_t *tmpidx, uint32_t cap) {
    pdl_enter();
    const uint32_t i0 = blockIdx.x * (SC_BLOCK * SC_PLACE_ILP) + threadIdx.x;
    uint32_t c[SC_PLACE_ILP], sl[SC_PLACE_ILP], st[SC_PLACE_ILP];
    // keys are requested before the live count is known (see k_prepass)
#pragma unroll
    for (int u = 0; u < SC_PLACE_ILP; ++u) {
        const uint32_t i = i0 + u * SC_BLOCK;
        c[u] = SC_INVALID_CELL;
        if (i < cap) c[u] = cell_key[i];
    }
    // the same bound key_particle counted under (see the invariant there)
    const uint32_t n = cnt->n < cap ? cnt->n : cap;
#pragma unroll
    for (int u = 0; u < SC_PLACE_ILP; ++u)
        if (i0 + u * SC_BLOCK >= n) c[u] = SC_INVALID_CELL;
#pragma unroll
    for (int u = 0; u < SC_PLACE_ILP; ++u)
        if (c[u] != SC_INVALID_CELL) {
            st[u] = cell_start[c[u]];
            sl[u] = atomicSub(&cell_count[c[u]], 1u) - 1u;
        }
#pragma unroll
    for (int u = 0; u < SC_PLACE_ILP; ++u)
        if (c[u] != SC_INVALID_CELL) tmpidx[st[u] + sl[u]] = i0 + u * SC_BLOCK;
}

// K3: rank inside the cell by (x, uid) and gather the particle record to its final sorted position.
// Produces exactly np.lexsort((x, floor(y / d))) (collision_detector.py:127) as the concatenation of cells.
// kEns: the grid is the members' grids stacked (Members); a cell row is then a row of its member's grid
template <typename Real, bool kEns = false>
__global__ void __launch_bounds__(SC_BLOCK)
k_rank_gather(Counters *cnt, Grid g, const uint32_t *cell_start, const uint32_t *tmpidx,
              const uint32_t *cell_key, const double2 *pos,
              const typename Vec2<Real>::type *vel, const uint32_t *uid,
              const uint32_t *wall_bits, const uint32_t *wall_slot,
              double2 *pos_s, float2 *rel_s,
              typename Vec2<Real>::type *vel_s, uint32_t *uid_s,
              uint32_t *cell_key_s, uint32_t *wall_bits_s,
              uint32_t *wall_slot_s, SearchRec *rec_s, BlockDesc *desc, Members E) {
    pdl_enter();
    const uint32_t n = cell_start[g.ncells];
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    // the density kernel's per-tick counters (read by sc_debug_untiled_blocks after the tick, so not reset any later)
    if (t == 0) { cnt->pair_cursor = 0; cnt->n_untiled = 0; }
    if (t >= n) return;
    const uint32_t i = tmpidx[t];
    const uint32_t c = cell_key[i];
    const uint32_t beg = cell_start[c], end = cell_start[c + 1];
    const double2 p = pos[i];
    const uint32_t u = uid[i];
    // the rest of the record: independent gathers, issued before the ranking walk so that they overlap its chain
    const typename Vec2<Real>::type v_own = vel[i];
    const bool touching = (wall_bits[i >> 5] >> (i & 31)) & 1u;
    const uint32_t um = u & 0x7FFFFFFFu;  // ties are broken by identity; bit 31 only marks a ghost copy
    // Two records of one identity at one x never meet in a correct run, but if they do (a uid handed to set_state_uids
    // twice, a strip exchange that keeps a migrant or a ghost it should drop) the array index decides: the ranks must
    // stay a permutation of the cell.  Two equal ranks would leave a sorted slot unwritten, and the pair kernels would
    // then walk the cell neighborhood of whatever stale cell key that slot held - outside the arrays.
    uint32_t rank = 0;
    for (uint32_t m = beg; m < end; ++m) {
        if (m == t) continue;
        const uint32_t j = tmpidx[m];
        const double xj = pos[j].x;
        const uint32_t uj = uid[j] & 0x7FFFFFFFu;
        rank += (x_less(xj, p.x) || (!x_less(p.x, xj) && (uj < um || (uj == um && j < i)))) ? 1u : 0u;
    }
    const uint32_t f = beg + rank;
    pos_s[f] = p;
    {   // cell-relative fp32 copy for the pair kernels' screening (see collect_neighbors)
        uint32_t cr = c / (uint32_t)g.ncols;
        const uint32_t cc = c - cr * (uint32_t)g.ncols;
        if constexpr (kEns) cr %= (uint32_t)E.nrows;
        float2 r;
        r.x = (float)(p.x - (double)((int)cc + g.col_min) * g.d);
        r.y = (float)(p.y - (double)((int)cr + g.row_min) * g.d);
        rel_s[f] = r;
        // the tiled pair kernels read position, cell column and identity as one 16-byte record (sc_tile.cuh)
        if (rec_s) rec_s[f] = make_float4(r.x, r.y, (float)cc, __uint_as_float(u));
    }
    if (desc) {  // the block of the tiled pair kernels this particle opens / closes: its three windows (sc_tile.cuh)
        const uint32_t nc = (uint32_t)g.ncols;
        if ((f & (SC_TILE - 1u)) == 0u)
            reinterpret_cast<uint4 *>(desc + f / SC_TILE)[0] =
                make_uint4(cell_start[c - 1u], cell_start[c + nc - 1u], cell_start[c - nc - 1u], c);
        if ((f & (SC_TILE - 1u)) == SC_TILE - 1u || f == n - 1u)
            reinterpret_cast<uint4 *>(desc + f / SC_TILE)[1] =
                make_uint4(cell_start[c + 2u], cell_start[c + nc + 2u], cell_start[c - nc + 2u], c);
    }
    vel_s[f] = v_own;
    uid_s[f] = u;
    cell_key_s[f] = c;
    if (touching) {
        wall_slot_s[f] = wall_slot[i];
        atomicOr(&wall_bits_s[f >> 5], 1u << (f & 31));
    }
}

// ------------------------------------------------------------------------------------------------------------
// uid -> rank among live particles (= the reference's row index, crate.py:146-159)
__global__ void __launch_bounds__(SC_BLOCK)
k_mark_alive(const uint32_t *n_ptr, const uint32_t *uid, uint32_t *alive) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    alive[uid[s]] = 1u;
}

// neighbor counts (and optionally lists, as sorted indices) - the parity tap and the SC_NOISE_HOST split step
__global__ void __launch_bounds__(SC_BLOCK)
k_count_neighbors(Counters *cnt, Grid g, const uint32_t *cell_start,
                  const double2 *pos, const float2 *rel,
                  const uint32_t *cell_key, const uint32_t *uid,
                  const uint32_t *rank_of_uid, uint32_t *count_by_rank,
                  uint32_t *list_sorted) {
    const uint32_t n = cell_start[g.ncells];
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    __shared__ uint32_t s_list[SC_MAX_NEIGHBORS * SC_BLOCK];
    NbrList lst{s_list + threadIdx.x};
    const int K = collect_neighbors(s, cell_key[s], g, cell_start, rel, pos, lst);
    if (list_sorted)
        for (int k = 0; k < K; ++k) list_sorted[(size_t)s * SC_MAX_NEIGHBORS + k] = lst.get(k) & SC_IDX_MASK;
    count_by_rank[rank_of_uid[uid[s]]] = (uint32_t)K;
    atomicAdd(&cnt->n_pairs, (uint32_t)K);
}

// sum of the per-particle pair counts of the last tick (on demand: the step itself keeps no running total)
__global__ void __launch_bounds__(SC_BLOCK)
k_sum_pair_counts(const uint32_t *n_ptr, const uint8_t *pair_cnt, uint32_t *total) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t v = s < *n_ptr ? pair_cnt[s] : 0u;
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(total, v);
}

// ---- scatter from sorted order to original (rank) order for host-visible arrays -------------------------------
template <typename T2>
__global__ void __launch_bounds__(SC_BLOCK)
k_scatter_vec2(const uint32_t *n_ptr, const uint32_t *uid,
               const uint32_t *rank_of_uid, const T2 *src, double2 *dst) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    const T2 v = src[s];
    double2 o;
    o.x = (double)v.x; o.y = (double)v.y;
    dst[rank_of_uid[uid[s]]] = o;
}
template <typename T>
__global__ void __launch_bounds__(SC_BLOCK)
k_scatter_scalar(const uint32_t *n_ptr, const uint32_t *uid,
                 const uint32_t *rank_of_uid, const T *src, double *dst) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    dst[rank_of_uid[uid[s]]] = (double)src[s];
}
// pressure / surface normal out of the packed PS records
template <typename Real>
__global__ void __launch_bounds__(SC_BLOCK)
k_scatter_ps(const uint32_t *n_ptr, const uint32_t *uid,
             const uint32_t *rank_of_uid, const PS<Real> *src, double *prs,
             double2 *tens) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    const PS<Real> v = src[s];
    const uint32_t r = rank_of_uid[uid[s]];
    if (prs) prs[r] = (double)v.p;
    if (tens) { double2 o; o.x = (double)v.sx; o.y = (double)v.sy; tens[r] = o; }
}
// positions in original order.  `wall_bits` (or NULL): the wall bitmap of a next tick whose hard-wall fix the force
// kernel already applied (NextKeys); a particle it moved is reported at its position before the fix, as the tick left it.
__global__ void __launch_bounds__(SC_BLOCK)
k_scatter_pos(const uint32_t *n_ptr, const uint32_t *uid, const uint32_t *rank_of_uid, const double2 *pos,
              const uint32_t *wall_bits, const uint32_t *wall_slot, const double2 *wall_pre, double2 *dst) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    const bool fixed = wall_bits && ((wall_bits[s >> 5] >> (s & 31)) & 1u);
    dst[rank_of_uid[uid[s]]] = fixed ? wall_pre[wall_slot[s]] : pos[s];
}
__global__ void __launch_bounds__(SC_BLOCK)
k_scatter_uid(const uint32_t *n_ptr, const uint32_t *uid,
              const uint32_t *rank_of_uid, uint32_t *dst) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    dst[rank_of_uid[uid[s]]] = uid[s];
}

// search taps: rows_sorted[s] = floor(y / d) of the particle at sorted index s, order[s] = its original index
__global__ void __launch_bounds__(SC_BLOCK)
k_tap_search(const uint32_t *n_ptr, Grid g, const double2 *pos,
             const uint32_t *uid, const uint32_t *rank_of_uid,
             long long *rows_sorted, long long *order) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    rows_sorted[s] = (long long)floor(pos[s].y / g.d);
    order[s] = (long long)rank_of_uid[uid[s]];
}

// neighbor lists in original index order holding original indices, -1 padded (collision_detector.py:46-48)
__global__ void __launch_bounds__(SC_BLOCK)
k_tap_lists(const uint32_t *n_ptr, const uint32_t *uid,
            const uint32_t *rank_of_uid, const uint32_t *count_by_rank,
            const uint32_t *list_sorted, int *idx_out) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    const uint32_t r = rank_of_uid[uid[s]];
    const uint32_t K = count_by_rank[r];
    for (uint32_t k = 0; k < SC_MAX_NEIGHBORS; ++k)
        idx_out[(size_t)r * SC_MAX_NEIGHBORS + k] =
            k < K ? (int)rank_of_uid[uid[list_sorted[(size_t)s * SC_MAX_NEIGHBORS + k]]] : -1;
}

// wall contact counts V_i (crate.py:229-232) in original order
__global__ void __launch_bounds__(SC_BLOCK)
k_tap_wall_counts(const uint32_t *n_ptr, DevParams P, const __grid_constant__ WallParams W,
                  const uint32_t *uid, const uint32_t *rank_of_uid,
                  const uint32_t *wall_bits, const uint32_t *wall_slot,
                  const double2 *wall_pre, int *out) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *n_ptr) return;
    int V = 0;
    if ((wall_bits[s >> 5] >> (s & 31)) & 1u) {
        const double2 pre = wall_pre[wall_slot[s]];
        for (int q = 0; q < W.S; ++q) {
            double cx, cy;
            if (point_segment(pre.x, pre.y, W.seg[q][0], W.seg[q][1], W.seg[q][2], W.seg[q][3], cx, cy) <= P.touch) ++V;
        }
    }
    out[rank_of_uid[uid[s]]] = V;
}

// geometry_utils.py:7-39 as a dense P x S op (the reference's own unit test pins this one)
__global__ void __launch_bounds__(SC_BLOCK)
k_points_segments(const double2 *p, uint32_t P_, const double *seg, int S,
                  double *nearest, double *dist) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= P_ * (uint32_t)S) return;
    const uint32_t i = t / (uint32_t)S, q = t % (uint32_t)S;
    double cx, cy;
    dist[t] = point_segment(p[i].x, p[i].y, seg[4 * q], seg[4 * q + 1], seg[4 * q + 2], seg[4 * q + 3], cx, cy);
    nearest[2 * (size_t)t] = cx;
    nearest[2 * (size_t)t + 1] = cy;
}

// ------------------------------------------------------------------------------------------------------------
// create_new_particles (crate.py:138-147) + ParticleSource.generate_particles (particle_source.py:17-24) on the device,
// production mode: the emission count of each source was drawn on the host from the counter stream (no device data
// needed); HOW MANY of them fit - min(n, max_particles - particle_count), with particle_count the count BEFORE this
// tick's removal and after the earlier sources of this tick, exactly as the reference evaluates it - is decided here
// from the device-resident count, so the tick needs no host round trip.  One block; sources emit a handful per tick.
struct EmitSource { double px, py, radius, vx, vy, vnoise; unsigned long long key; uint32_t n, uid_base; };
struct EmitParams { EmitSource src[SC_MAX_SOURCES]; int nsrc; uint32_t max_particles; };
template <typename Real>
__global__ void __launch_bounds__(SC_BLOCK)
k_emit(Counters *cnt, const __grid_constant__ EmitParams E, double2 *pos, typename Vec2<Real>::type *vel, uint32_t *uid,
       uint32_t cap) {
    pdl_enter();
    __shared__ uint32_t s_base[SC_MAX_SOURCES], s_cnt[SC_MAX_SOURCES];
    if (threadIdx.x == 0) {
        uint32_t P = cnt->n;
        for (int q = 0; q < E.nsrc; ++q) {
            const uint32_t room = E.max_particles > P ? E.max_particles - P : 0u;
            uint32_t a = E.src[q].n < room ? E.src[q].n : room;
            if (P + a > cap) { a = cap > P ? cap - P : 0u; cnt->overflow = 1u; }
            s_base[q] = P; s_cnt[q] = a;
            P += a;
        }
        cnt->n = P;
    }
    __syncthreads();
    for (int q = 0; q < E.nsrc; ++q) {
        const EmitSource &S = E.src[q];
        for (uint32_t k = threadIdx.x; k < s_cnt[q]; k += blockDim.x) {
            const double ux = source_uniform(S.key, 1ull + 4ull * k), uy = source_uniform(S.key, 2ull + 4ull * k);
            const double wx = source_uniform(S.key, 3ull + 4ull * k), wy = source_uniform(S.key, 4ull + 4ull * k);
            const uint32_t at = s_base[q] + k;
            pos[at] = make_double2((ux - 0.5) * S.radius + S.px, (uy - 0.5) * S.radius + S.py);      // particle_source.py:21
            typename Vec2<Real>::type v;                                                            // particle_source.py:22-23
            v.x = (Real)(S.vx + (wx - 0.5) * S.vnoise);
            v.y = (Real)(S.vy + (wy - 0.5) * S.vnoise);
            vel[at] = v;
            uid[at] = S.uid_base + k;
        }
    }
}

// The same for the members of an ensemble (sc_ens_emit_particles).  Member m draws its own counts from its own stream
// (key: the member's seed) and is clamped against ITS live count: mcount[m], or - when a step ran since mcount was
// written (`from_scan`) - the member's share of that step's cell scan, which is its count after that tick's removal.  Its
// identities continue from next_local[m] and advance by the drawn count.  Everything the host draws travels in the
// launch's parameters (w = [max_particles | drawn counts members x nsrc] of members m0 .. m0 + members - 1), so no host
// buffer is copied per tick; members beyond one launch's parameter space go in further launches, each appending behind
// the last (the host caps the total, so the capacity test below never drops a particle).  One block, a thread per
// member, members in chunks of the block.
struct EnsEmitSource { double px, py, radius, vx, vy, vnoise; uint32_t index; };
struct EnsEmitHead {
    EnsEmitSource src[SC_MAX_SOURCES];
    int nsrc, from_scan;
    uint32_t m0, members, uid_bits, ncells;  // ncells: cells of one member's grid
    unsigned long long tick;
};
template <int kWords> struct EnsEmitParams { EnsEmitHead h; uint32_t w[kWords]; };
#define SC_EMIT_WORDS_SMALL 256   // launches whose draws fit 1 KB pay for no more parameter space
#define SC_EMIT_WORDS 7936        // the largest that keeps the parameters within the 32 764 bytes a launch may take
static_assert(sizeof(EnsEmitParams<SC_EMIT_WORDS>) <= 32764, "kernel parameter space");
#define SC_EMIT_THREADS 1024
template <typename Real, int kWords>
__global__ void __launch_bounds__(SC_EMIT_THREADS)
k_emit_members(Counters *cnt, const __grid_constant__ EnsEmitParams<kWords> E, uint32_t *next_local,
               const unsigned long long *seed, uint32_t *mcount, const uint32_t *cell_start, double2 *pos,
               typename Vec2<Real>::type *vel, uint32_t *uid, uint32_t cap) {
    pdl_enter();
    const uint32_t M = E.h.members;
    const uint32_t *maxp = E.w, *draw = E.w + M;
    const uint32_t n0 = cnt->n;
    uint32_t run = 0;  // particles placed by the chunks before
    for (uint32_t c0 = 0; c0 < M; c0 += SC_EMIT_THREADS) {
        const uint32_t j = c0 + threadIdx.x, m = E.h.m0 + j;
        uint32_t a[SC_MAX_SOURCES], mine = 0;
        if (j < M) {
            uint32_t P = E.h.from_scan ? cell_start[(size_t)(m + 1) * E.h.ncells] - cell_start[(size_t)m * E.h.ncells] : mcount[m];
            for (int q = 0; q < E.h.nsrc; ++q) {
                const uint32_t room = maxp[j] > P ? maxp[j] - P : 0u, n = draw[(size_t)j * E.h.nsrc + q];
                a[q] = n < room ? n : room;
                P += a[q];
                mine += a[q];
            }
            mcount[m] = P;
        }
        uint32_t total;
        const uint32_t before = block_exclusive_scan_n<SC_EMIT_THREADS>(mine, total);
        if (j < M) {
            const uint64_t tkey = tick_key(seed[m], E.h.tick);
            uint32_t at = n0 + run + before, local = next_local[m];
            for (int q = 0; q < E.h.nsrc; ++q) {
                const EnsEmitSource &S = E.h.src[q];
                const uint64_t key = source_key(tkey, S.index);
                for (uint32_t k = 0; k < a[q]; ++k, ++at) {
                    if (at >= cap) { cnt->overflow = 1u; break; }
                    const double ux = source_uniform(key, 1ull + 4ull * k), uy = source_uniform(key, 2ull + 4ull * k);
                    const double wx = source_uniform(key, 3ull + 4ull * k), wy = source_uniform(key, 4ull + 4ull * k);
                    pos[at] = make_double2((ux - 0.5) * S.radius + S.px, (uy - 0.5) * S.radius + S.py);   // as k_emit
                    typename Vec2<Real>::type v;
                    v.x = (Real)(S.vx + (wx - 0.5) * S.vnoise);
                    v.y = (Real)(S.vy + (wy - 0.5) * S.vnoise);
                    vel[at] = v;
                    uid[at] = (m << E.h.uid_bits) | (local + k);
                }
                local += draw[(size_t)j * E.h.nsrc + q];
            }
            next_local[m] = local;
        }
        run += total;
    }
    __syncthreads();
    if (threadIdx.x == 0) cnt->n = n0 + run < cap ? n0 + run : cap;
}

// per-member live counts: mcount[m], refreshed from the last step's cell scan when `from_scan`; copied to `out` (or NULL)
__global__ void __launch_bounds__(SC_BLOCK)
k_member_counts(uint32_t M, uint32_t ncells, int from_scan, const uint32_t *cell_start, uint32_t *mcount, uint32_t *out) {
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const uint32_t v = from_scan ? cell_start[(size_t)(m + 1) * ncells] - cell_start[(size_t)m * ncells] : mcount[m];
    mcount[m] = v;
    if (out) out[m] = v;
}

// min / max cell coordinates of an arbitrary point set (standalone detect_particle_collisions)
__global__ void __launch_bounds__(SC_BLOCK)
k_cell_bounds(const double2 *pos, uint32_t n, double d, int *bounds /* rmin rmax cmin cmax */) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double fr = floor(pos[i].y / d), fc = floor(pos[i].x / d);
    const int r = (fr >= -2.0e9 && fr <= 2.0e9) ? (int)fr : 0, c = (fc >= -2.0e9 && fc <= 2.0e9) ? (int)fc : 0;
    atomicMin(&bounds[0], r); atomicMax(&bounds[1], r);
    atomicMin(&bounds[2], c); atomicMax(&bounds[3], c);
}

__global__ void __launch_bounds__(SC_BLOCK) k_iota(uint32_t *a, uint32_t base, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = base + i;
}

// COLD start of a tick (the first tick of a context, the first after the cell grid was rebuilt), as a launch of its own:
// zero the cell-count grid, the tick's wall bitmaps and the scan's descriptors, reset the counters.  `carry` (or NULL):
// the last scan's total, = the live count when no force kernel carried it.
// The same launch, with `restore`, takes back what the last force kernel did for a next tick that will not use it
// (NextKeys, dropped by the host): the positions of the particles it moved in the hard-wall fix are put back from the
// wall side list (bits_a = that tick's wall bitmap) before the bitmaps are zeroed.
struct KeyRestore { double2 *pos; const uint32_t *wall_slot; const double2 *wall_pre; };
__global__ void __launch_bounds__(SC_BLOCK)
k_begin_tick(Counters *cnt, uint32_t *cell_count, uint32_t ncells, const uint32_t *carry,
             uint32_t *bits_a, uint32_t *bits_b, uint32_t nbits_words,
             unsigned long long *scan_desc, uint32_t scan_words, uint32_t cap, KeyRestore restore) {
    pdl_enter();
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    if (tid == 0) {
        if (carry) cnt->n = *carry;
        if (cnt->n > cap) { cnt->n = cap; cnt->overflow = 1u; }
        cnt->n_wall[0] = 0; cnt->n_wall[1] = 0; cnt->n_pairs = 0; cnt->pair_cursor = 0; cnt->n_untiled = 0;
    }
    uint4 *c4 = reinterpret_cast<uint4 *>(cell_count);
    const uint32_t n4 = ncells / 4;
    for (uint32_t i = tid; i < n4; i += nth) c4[i] = make_uint4(0, 0, 0, 0);
    for (uint32_t i = n4 * 4 + tid; i < ncells; i += nth) cell_count[i] = 0;
    for (uint32_t i = tid; i < nbits_words; i += nth) {
        if (restore.pos)  // a set bit is a particle the wall fix moved (only the key pass sets them; K4 zeroed the rest)
            for (uint32_t m = bits_a[i]; m; m &= m - 1u) {
                const uint32_t k = i * 32u + (uint32_t)(__ffs(m) - 1);
                restore.pos[k] = restore.wall_pre[restore.wall_slot[k]];
            }
        bits_a[i] = 0; bits_b[i] = 0;
    }
    for (uint32_t i = tid; i < scan_words; i += nth) scan_desc[i] = 0ull;  // tile descriptors + ticket of the cell scan
}

template <typename Real>
__global__ void __launch_bounds__(SC_BLOCK)
k_convert_vel_in(const double2 *src, typename Vec2<Real>::type *dst, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    typename Vec2<Real>::type v;
    v.x = (Real)src[i].x; v.y = (Real)src[i].y;
    dst[i] = v;
}

}  // namespace sc
