// sc_tile.cuh - the mixed-precision pair kernels: K4 and K5 with the neighborhood of a block staged in shared memory.
//
// A block owns SC_TILE consecutive particles of the sorted set.  Because the sort is cell-major (row, col, x), every
// neighbor of those particles lies in one of three CONTIGUOUS windows of the sorted set - the block's own stretch of
// its cell row(s) widened by one cell at each end, and the same stretch of cells one row below / one row above:
//
//     W0 = [cell_start[c_lo - 1],         cell_start[c_hi + 2])           same row(s)
//     W1 = [cell_start[c_lo + ncols - 1], cell_start[c_hi + ncols + 2])   next row(s)
//     W2 = [cell_start[c_lo - ncols - 1], cell_start[c_hi - ncols + 2])   previous row(s)
//
// (c_lo, c_hi = cells of the block's first / last particle; k_rank_gather leaves the six bounds in a per-block
// descriptor, so the kernel starts with ONE dependent load instead of a chain of four).  The windows and the block's
// slice of the cell boundaries are copied into shared memory with coalesced loads; the candidate loop then reads
// 16-byte records (cell-relative position, cell column, uid) from shared memory instead of issuing a dependent global
// load per candidate.  A staged particle is addressed by its position in the concatenation W0 | W1 | W2 ("local
// index", 11 bits), so the per-thread neighbor lists are 16-bit.
//
// When the three windows do not fit the staging buffer (a block of spray that spans many sparse rows), the block
// runs the same code with a pass-through accessor: local index = sorted index, reads go to global memory.  The
// arithmetic is identical in both modes, so a particle's result does not depend on which mode its block ran in
// (the strip decomposition relies on that: a ghost and its owner must compute the same bits).
//
// The neighbor search is the one of k_density in sc_pair.cuh (same reference lines, same list order, same 20-trim, same
// fp32-screen / fp64-replay acceptance); only the data movement differs, and the pair geometry is fp32.  Measured on
// B200 (dam-break 1M) against an fp32 K4 that gathered from global memory: 69 -> 59 us.  K5 (k_force_tile) reads the
// neighbors' pressure, normal and velocity from the same staged windows.
#pragma once
#include "sc_pair.cuh"

namespace sc {

#define SC_TILE_CAP (5 * SC_TILE)              // staged particles per block (3 windows of ~SC_TILE + a few cells each)
#ifndef SC_K5_ROWS
#define SC_K5_ROWS 6                           // pair-record slots of a block that K5 stages in shared memory
#endif
#define SC_TILE_CELLS (SC_TILE + SC_TILE / 2 + 64)  // staged cell boundaries per row (blocks that wrap around a row end
                                               // read them from global)

// search record of one sorted particle, written by k_rank_gather in mixed mode:
//   x, y = cell-relative position (see collect_neighbors), z = (float)cell column, w = uid bits
// The column travels as a float so that the x offset between two cells is one subtraction and one FMA:
//   x_j - x_i = (rel_j.x - rel_i.x) + (col_j - col_i) * d     with col_j - col_i in {-1, 0, 1}, exact in fp32.
typedef float4 SearchRec;

// Per block of SC_TILE sorted particles, written by k_rank_gather (the threads that place the block's first and last
// particle): the three windows and the block's first / last cell.  One 32-byte read replaces a chain of dependent
// loads (particle count -> cell keys -> cell boundaries) at the head of K4 and K5.
struct __align__(16) BlockDesc {
    uint32_t base[3], c_lo;  // first sorted index of W0, W1, W2
    uint32_t end[3], c_hi;   // one past the last
};

struct TileWindows {
    uint32_t base[3];  // first STAGED sorted index of W0, W1, W2: the window's first index rounded down to even, so that
                       // 8-byte arrays (velocities) start 16-byte aligned, which the bulk copy needs
    uint32_t off[3];   // first local index of W0, W1, W2 (staged) / = base (pass-through)
    uint32_t cnt[3];   // staged particles per window (even)
    uint32_t total;    // staged particles
    uint32_t c_lo, ncw;  // first cell of the block, cells per row slice (c_lo - 1 .. c_hi + 2)
    bool staged, cells_staged;
};

__device__ __forceinline__ TileWindows tile_windows(const BlockDesc *desc) {
    const uint4 lo = reinterpret_cast<const uint4 *>(desc)[0], hi = reinterpret_cast<const uint4 *>(desc)[1];
    TileWindows w;
    w.base[0] = lo.x & ~1u; w.base[1] = lo.y & ~1u; w.base[2] = lo.z & ~1u; w.c_lo = lo.w;
    w.cnt[0] = (hi.x - w.base[0] + 1u) & ~1u; w.cnt[1] = (hi.y - w.base[1] + 1u) & ~1u; w.cnt[2] = (hi.z - w.base[2] + 1u) & ~1u;
    w.total = w.cnt[0] + w.cnt[1] + w.cnt[2];
    w.ncw = hi.w - lo.w + 4u;
    w.staged = w.total <= SC_TILE_CAP;
    w.cells_staged = w.staged && w.ncw <= SC_TILE_CELLS;
    if (w.staged) { w.off[0] = 0u; w.off[1] = w.cnt[0]; w.off[2] = w.cnt[0] + w.cnt[1]; }
    else { w.off[0] = w.base[0]; w.off[1] = w.base[1]; w.off[2] = w.base[2]; }
    return w;
}

// ---- bulk copies (TMA engine, no tensor map): global -> shared, completion counted in bytes on an mbarrier ----------
// One elected thread arms the barrier with the byte total and issues the copies; every thread then waits on the
// barrier's phase.  No thread spends an instruction on moving the data, no registers hold it in flight, and the wait
// replaces the __syncthreads of a load/store staging loop.  Source, destination and size must be multiples of 16 bytes.
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");  // visible to the async proxy
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// the same, made opaque to the compiler: on sm_100 a shared address is (cluster CTA rank << 24) + offset, and nvcc would
// rather re-derive it (S2UR SR_CgaCtaId; UMOV; ULEA: three issue slots) inside a hot loop than keep it in a register
__device__ __forceinline__ uint32_t smem_addr_pinned(const void *p) {
    uint32_t a = smem_addr(p);
    asm volatile("" : "+r"(a));
    return a;
}

// the three windows of a `stride`-byte-per-particle array into shared memory at `dst` (W0 | W1 | W2); returns bytes
__device__ __forceinline__ uint32_t stage_windows(const TileWindows &w, const void *src, uint32_t stride, uint32_t dst,
                                                  uint32_t bar) {
    const char *g = reinterpret_cast<const char *>(src);
#pragma unroll
    for (int q = 0; q < 3; ++q)
        if (w.cnt[q]) bulk_g2s(dst + w.off[q] * stride, g + (size_t)w.base[q] * stride, w.cnt[q] * stride, bar);
    return w.total * stride;
}

// accessors: shared memory by 32-bit shared address (keeps the address arithmetic to one instruction), or global
template <typename T> struct SmemAcc {
    uint32_t addr;
    __device__ __forceinline__ T get(uint32_t L) const;
    // a CURSOR walks the staged array by byte address, so that the candidate loop's load needs no address arithmetic
    static constexpr uint32_t kStep = (uint32_t)sizeof(T);
    __device__ __forceinline__ uint32_t cursor(uint32_t L) const { return addr + L * kStep; }
    __device__ __forceinline__ uint32_t index(uint32_t cur) const { return (cur - addr) / kStep; }
    __device__ __forceinline__ T at(uint32_t cur) const;
};
template <> __device__ __forceinline__ float4 SmemAcc<float4>::get(uint32_t L) const {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr + L * 16u));
    return v;
}
template <> __device__ __forceinline__ float4 SmemAcc<float4>::at(uint32_t cur) const {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(cur));
    return v;
}
template <> __device__ __forceinline__ uint2 SmemAcc<uint2>::get(uint32_t L) const {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr + L * 8u));
    return v;
}
template <> __device__ __forceinline__ float2 SmemAcc<float2>::get(uint32_t L) const {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr + L * 8u));
    return v;
}
template <typename T> struct GmemAcc {
    const T *p;
    __device__ __forceinline__ T get(uint32_t L) const { return p[L]; }
    static constexpr uint32_t kStep = 1u;
    __device__ __forceinline__ uint32_t cursor(uint32_t L) const { return L; }
    __device__ __forceinline__ uint32_t index(uint32_t cur) const { return cur; }
    __device__ __forceinline__ T at(uint32_t cur) const { return p[cur]; }
};
// per-thread neighbor list, one column per thread; 16-bit entries when the indices are local (11 bits + row code)
template <typename E, int kShift> struct TileList {
    E *col;
    __device__ __forceinline__ void set(int k, uint32_t L, uint32_t code) { col[k * SC_TILE] = (E)(L | (code << kShift)); }
    __device__ __forceinline__ void get(int k, uint32_t &L, uint32_t &code) const {
        const uint32_t e = col[k * SC_TILE];
        L = e & ((1u << kShift) - 1u); code = e >> kShift;
    }
};

__device__ __forceinline__ float rsqrt_ftz(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float sqrt_ftz(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// ------------------------------------------------------------------------------------------------------------
// The record K4 hands to K5 for each directed pair (i <- j): ONE 8-byte word.
//   .x  the SMALLER-magnitude component m of the unit vector n_ij, as a full fp32
//   .y  bits 0..27  the neighbor's index L in the block's frame (staged block: position in W0 | W1 | W2; pass-through
//                   block: sorted index) - K4 and K5 cut the sorted set into the same blocks and windows, so K5 reads
//                   its neighbor's (p, s, v) from shared memory at L with no translation
//       bit 28      which component m is (0: n.x, 1: n.y)
//       bit 29      sign of the other component, whose magnitude K5 restores as sqrt(1 - m^2) (>= 0.707: well conditioned)
// The vector K5 sees is good to ~1e-7 (fp32 grade).  Round 1 packed it as two signed 16-bit fractions (1.5e-5 per
// component): that was 250x coarser than the arithmetic around it and showed in the per-tick velocity INCREMENT.
__device__ __forceinline__ uint2 pair_encode(uint32_t L, float nx, float ny) {
    const bool y_small = fabsf(ny) < fabsf(nx);
    const float m = y_small ? ny : nx, big = y_small ? nx : ny;
    return make_uint2(__float_as_uint(m), L | (y_small ? 0x10000000u : 0u) | ((__float_as_uint(big) >> 2) & 0x20000000u));
}
__device__ __forceinline__ void pair_decode(uint2 r, uint32_t &L, float &nx, float &ny) {
    const float m = __uint_as_float(r.x);
    float big = sqrt_ftz(fmaf(-m, m, 1.0f));
    big = __uint_as_float(__float_as_uint(big) | ((r.y << 2) & 0x80000000u));
    const bool y_small = (r.y & 0x10000000u) != 0u;
    nx = y_small ? big : m;
    ny = y_small ? m : big;
    L = r.y & SC_IDX_MASK;
}

// SC_NOISE_HOST: the reference's noise stream.  Pair k of the particle with uid u takes the uniforms
// u[2 (off[rank_of_uid[u]] + k) + {0, 1}]: off holds CSR offsets in original index order (sc_step_finish) and is only
// valid until the next count kernel overwrites it.
struct HostNoise { const double *u; const uint32_t *off, *rank_of_uid; };
// ------------------------------------------------------------------------------------------------------------
// K4 body for one particle.  s = sorted index; b[] = the six boundaries of its four candidate ranges as LOCAL
// indices (m0, m3 | n0, n3 | p0, p3 of collect_neighbors, shifted into the staged windows).  List order = reference
// list order.
// kEns: the pair geometry and pressure take the particle's member's parameters and noise (Members); the search only
// depends on the diameter, which all members share
template <int kNoise, bool kEns, class Acc, class List>
__device__ __forceinline__ void density_particle(const Acc &A, List lst, const TileWindows &w, bool live, uint32_t s,
                                                 const uint32_t (&b)[6], const Grid &g, const DevParams &P,
                                                 const double2 *pos, uint2 *pair_rec,
                                                 uint8_t *pair_cnt, PS<float> *ps_out, const HostNoise &hn,
                                                 const Members &E) {
    const float df = P.f_d;
    const uint32_t d0 = w.off[0] - w.base[0], d1 = w.off[1] - w.base[1], d2 = w.off[2] - w.base[2];
    int K = 0;
    SearchRec me = make_float4(0, 0, 0, 0);
    if (live) {
        const float hi = P.f_band_hi, lo = P.f_band_lo;
        const uint32_t Ls = s + d0;
        me = A.get(Ls);
        int count = 0;
        // FIRST .. STOP (exclusive) in local indices, walking by STEP; BY = y of this particle in the frame of the
        // range's cell row; DELTA = local - sorted index of the range's window.  The walk is on a CURSOR (the staged
        // record's shared-memory byte address), so the loop's load needs no address arithmetic: 15 instructions per
        // rejected candidate instead of 20.
        // (Ending the walk once a candidate is more than d away in x - rows are sorted by x - was measured: the extra
        // predicate costs what the shorter walks save.  ONE loop over the four ranges with a range-switch inside - fewer
        // iterations per warp: max of sums instead of sum of maxes - was measured too: 71 us against 53, the switch
        // makes every iteration divergent.)
#define SC_TILE_RANGE(FIRST, STOP, STEP, BY, DR, DELTA, ASC)                                                     \
        {                                                                                                        \
            const float by = (BY);                                                                               \
            const uint32_t stop = A.cursor(STOP);                                                                \
            /* trim_collisions (collision_detector.py:91-93): the 20th accept moves the cursor to the end of the */ \
            /* range (no `break`, which keeps the warp from reconverging; no count test in the loop condition) */ \
            if (count < SC_MAX_NEIGHBORS)                                                                        \
            for (uint32_t cur = A.cursor(FIRST); cur != stop; cur += (STEP) * Acc::kStep) {                     \
                const SearchRec r = A.at(cur);                                                                   \
                const float dx = fmaf(r.z - me.z, df, r.x - me.x), dy = r.y - by;                                \
                const float qd = fmaf(dx, dx, dy * dy);                                                          \
                /* qd > hi: surely farther than d (NaN too: the reference rejects NaN); qd < lo: surely inside */ \
                if (qd <= hi) {                                                                                  \
                    const uint32_t L = A.index(cur);                                                             \
                    if (qd < lo || accept_exact(pos[s], pos[L - (DELTA)], g.d, (DR), (ASC))) {                   \
                        lst.set(count, L, (uint32_t)((DR) + 1));                                                 \
                        if (++count == SC_MAX_NEIGHBORS) cur = stop - (STEP) * Acc::kStep;                       \
                    }                                                                                            \
                }                                                                                                \
            }                                                                                                    \
        }
        SC_TILE_RANGE(Ls + 1u, b[1], 1u, me.y, 0, d0, true)
        SC_TILE_RANGE(b[2], b[3], 1u, me.y - df, 1, d1, true)
        SC_TILE_RANGE(Ls - 1u, b[0] - 1u, 0xFFFFFFFFu, me.y, 0, d0, false)
        SC_TILE_RANGE(b[5] - 1u, b[4] - 1u, 0xFFFFFFFFu, me.y + df, -1, d2, false)
#undef SC_TILE_RANGE
        K = count;
    }
    // Records are SLOT-MAJOR inside the block's own region of the pair buffer: record k of thread t sits at
    // (block * 20 + k) * SC_TILE + t.  No allocation (no scan, no atomic, no offset array), a warp's stores of one slot
    // are one contiguous 256-byte run, and K5 can bulk-copy the first slots of the whole block without knowing anything.
    if (!live) return;
    pair_cnt[s] = (uint8_t)K;
    const uint32_t uid_s = __float_as_uint(me.w);
    DevParams Pm;
    if constexpr (kEns) Pm = member_params(E, uid_s);
    const DevParams &PP = pick_params<kEns>(P, Pm);
    const float inv_d = P.f_inv_d;
    const float amp = PP.f_amp;
    uint32_t nbase = 0u;
    if constexpr (kNoise == SC_NOISE_HOST) nbase = hn.off[hn.rank_of_uid[uid_s]];
    float ax = 0, ay = 0, psum = 0;
    uint2 *out = pair_rec + (size_t)blockIdx.x * (SC_MAX_NEIGHBORS * SC_TILE) + threadIdx.x;
    for (int k = 0; k < K; ++k) {
        uint32_t L, code;  // code = dr + 1
        lst.get(k, L, code);
        const SearchRec r = A.get(L);
        float rx = fmaf(me.z - r.z, df, me.x - r.x);
        float ry = (me.y - r.y) - fmaf((float)code, df, -df);  // the neighbor's row is dr * d further down
        // crate.py:167-174: the neighbor's position is noised, then the unit vector from it to i and the distance
        if constexpr (kNoise == SC_NOISE_COUNTER) {
            if (!kEns || PP.noise_mode == SC_NOISE_COUNTER) {
                float fx, fy;  // uniforms + 1
                pair_noise_f32_1to2(pair_noise_bits(PP.tick_key, noise_uid<kEns>(E, uid_s),
                                                    noise_uid<kEns>(E, __float_as_uint(r.w))), fx, fy);
                rx = fmaf(1.5f - fx, amp, rx);  // 0.5 - u, exact
                ry = fmaf(1.5f - fy, amp, ry);
            }
        } else if constexpr (kNoise == SC_NOISE_HOST) {
            const size_t q = 2 * (size_t)(nbase + (uint32_t)k);
            const float ux = (float)hn.u[q], uy = (float)hn.u[q + 1];
            rx = fmaf(0.5f - ux, amp, rx);
            ry = fmaf(0.5f - uy, amp, ry);
        }
        const float q = fmaf(rx, rx, ry * ry);
        const float inv = rsqrt_ftz(q);
        const float nx = rx * inv, ny = ry * inv;
        const float cl = __saturatef((q * inv) * inv_d);  // np.clip(dist / d, 0, 1), crate.py:270
        const float wgt = 1.0f - cl;
        out[k * SC_TILE] = pair_encode(L, nx, ny);
        psum += wgt;
        const float c = cl * wgt;  // (1 - w) w, crate.py:340
        ax = fmaf(c, nx, ax);
        ay = fmaf(c, ny, ay);
    }
    float p = 0;
    if (K > 0) {
        const float pr = psum - PP.f_ignored;
        p = (pr > 0 || pr != pr) ? pr : 0.0f;  // np.maximum(0, pr), crate.py:273
    }
    PS<float> o;
    o.p = p; o.sx = ax; o.sy = ay; o.pad_ = 0;
    ps_out[s] = o;
}

#define SC_TILE_CELL_SLOTS (SC_TILE_CELLS + 8)  // a staged row slice starts at a multiple of 4 cells: up to 3 + 3 extra
#define SC_TILE_SMEM_K4 (SC_TILE_CAP * 16 + 3 * SC_TILE_CELL_SLOTS * 4 + SC_MAX_NEIGHBORS * SC_TILE * 2)

#ifndef SC_TILE_RESIDENT
#define SC_TILE_RESIDENT 1536  // threads per SM the register allocation is held to (1536 = 40 registers)
#endif
template <int kNoise, bool kEns = false>
__global__ void __launch_bounds__(SC_TILE, SC_TILE_RESIDENT / SC_TILE)
k_density_tile(Counters *cnt, Grid g, DevParams P, const uint32_t *cell_start,
               const BlockDesc *desc, const double2 *pos,
               const SearchRec *rec, const uint32_t *cell_key,
               uint2 *pair_rec, uint8_t *pair_cnt, PS<float> *ps_out, NextWallClear next,
               HostNoise hn, Members E) {  // last: the other parameters keep their offsets in every instantiation
    pdl_enter();
    clear_next_walls(next);
    // staged: [records 20 KB | cell boundaries 4.7 KB | 16-bit lists 10 KB]; pass-through: [32-bit lists 20 KB]
    __shared__ __align__(128) unsigned char s_raw[SC_TILE_SMEM_K4];
    __shared__ __align__(8) unsigned long long s_bar;
    static_assert(SC_TILE_SMEM_K4 >= SC_MAX_NEIGHBORS * SC_TILE * 4, "pass-through lists must fit");
    const uint32_t b0 = blockIdx.x * SC_TILE;
    const uint32_t s = b0 + threadIdx.x;
    // first round of loads, all independent: live count, block descriptor, own cell
    const uint32_t n = cell_start[g.ncells];
    if (b0 >= n) return;
    const TileWindows w = tile_windows(desc + blockIdx.x);
    const bool live = s < n;
    const uint32_t c = live ? cell_key[s] : w.c_lo;
    const uint32_t nc = (uint32_t)g.ncols;
    uint32_t b[6];
    if (w.staged) {
        SearchRec *s_rec = reinterpret_cast<SearchRec *>(s_raw);
        uint32_t *s_cs = reinterpret_cast<uint32_t *>(s_raw + SC_TILE_CAP * 16);
        uint16_t *s_list = reinterpret_cast<uint16_t *>(s_raw + SC_TILE_CAP * 16 + 3 * SC_TILE_CELL_SLOTS * 4);
        const uint32_t bar = smem_addr(&s_bar);
        // second round: the three windows and (unless the block wraps around a row end) its three slices of the cell
        // boundaries, by bulk copy.  A slice starts at the multiple of 4 cells at or below c_lo - 1 (16-byte alignment).
        const uint32_t i0 = w.c_lo - 1u, i1 = i0 + nc, i2 = i0 - nc;
        const uint32_t a0 = i0 & ~3u, a1 = i1 & ~3u, a2 = i2 & ~3u;
        if (threadIdx.x == 0) mbar_init(bar, 1u);
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t bytes = w.total * 16u;
            const uint32_t n0 = (i0 - a0 + w.ncw + 3u) & ~3u, n1 = (i1 - a1 + w.ncw + 3u) & ~3u, n2 = (i2 - a2 + w.ncw + 3u) & ~3u;
            if (w.cells_staged) bytes += (n0 + n1 + n2) * 4u;
            mbar_expect_tx(bar, bytes);
            stage_windows(w, rec, 16u, smem_addr(s_rec), bar);
            if (w.cells_staged) {
                const uint32_t cs = smem_addr(s_cs);
                bulk_g2s(cs, cell_start + a0, n0 * 4u, bar);
                bulk_g2s(cs + SC_TILE_CELL_SLOTS * 4u, cell_start + a1, n1 * 4u, bar);
                bulk_g2s(cs + 2u * SC_TILE_CELL_SLOTS * 4u, cell_start + a2, n2 * 4u, bar);
            }
        }
        const uint32_t d0 = w.off[0] - w.base[0], d1 = w.off[1] - w.base[1], d2 = w.off[2] - w.base[2];
        if (!w.cells_staged && live) {
            const uint32_t *cs0 = cell_start + c - 1u;
            b[0] = cs0[0] + d0; b[1] = cs0[3] + d0;
            b[2] = cs0[nc] + d1; b[3] = cs0[nc + 3u] + d1;
            b[4] = (cs0 - nc)[0] + d2; b[5] = (cs0 - nc)[3] + d2;
        }
        mbar_wait(bar, 0u);
        if (w.cells_staged) {
            const uint32_t q = c - w.c_lo;
            const uint32_t *r0 = s_cs + (i0 - a0) + q, *r1 = s_cs + SC_TILE_CELL_SLOTS + (i1 - a1) + q,
                           *r2 = s_cs + 2 * SC_TILE_CELL_SLOTS + (i2 - a2) + q;
            b[0] = r0[0] + d0; b[1] = r0[3] + d0;
            b[2] = r1[0] + d1; b[3] = r1[3] + d1;
            b[4] = r2[0] + d2; b[5] = r2[3] + d2;
        }
        density_particle<kNoise, kEns>(SmemAcc<SearchRec>{smem_addr_pinned(s_rec)}, TileList<uint16_t, 13>{s_list + threadIdx.x},
                                       w, live, s, b, g, P, pos, pair_rec, pair_cnt, ps_out, hn, E);
    } else {
        if (threadIdx.x == 0) atomicAdd(&cnt->n_untiled, 1u);  // rare; lets a test prove this path ran
        if (live) {
            const uint32_t *cs0 = cell_start + c - 1u;
            b[0] = cs0[0]; b[1] = cs0[3];
            b[2] = cs0[nc]; b[3] = cs0[nc + 3u];
            b[4] = (cs0 - nc)[0]; b[5] = (cs0 - nc)[3];
        }
        density_particle<kNoise, kEns>(GmemAcc<SearchRec>{rec},
                                       TileList<uint32_t, 28>{reinterpret_cast<uint32_t *>(s_raw) + threadIdx.x}, w,
                                       live, s, b, g, P, pos, pair_rec, pair_cnt, ps_out, hn, E);
    }
}

// ------------------------------------------------------------------------------------------------------------
// K5 (mixed mode): the same blocks and windows as K4.  The neighbors' pressure / surface normal
// (16 bytes) and velocity (8 bytes) are bulk-copied into shared memory while the threads fetch their own record
// offsets; the pair loop then reads ld.shared.v4 / .v2 at the local index the pair record carries, instead of two
// dependent global gathers per pair (which made a gathering K5 latency bound at 38 % occupancy).
// Round 1 built this with a load/store staging loop and measured it SLOWER than gathering (60 vs 46 us): the loop's
// instructions, its registers in flight and its barrier cost more than the gathers saved.  The bulk copy has none of
// the three.
template <bool kMonitor, bool kEns = false>
#ifndef SC_K5_TILE_MINBLOCKS
#define SC_K5_TILE_MINBLOCKS 4   // blocks per SM the register allocation is held to (4 = 64 registers)
#endif
__global__ void __launch_bounds__(SC_TILE, SC_K5_TILE_MINBLOCKS)
k_force_tile(const uint32_t *n_ptr, DevParams P0, const __grid_constant__ WallParams W, const BlockDesc *desc,
             const double2 *pos, const float2 *vel, const uint2 *pair_rec,
             const uint8_t *pair_cnt, const PS<float> *ps_in, const uint32_t *wall_bits, const uint32_t *wall_slot,
             const double2 *wall_pre, double2 *pos_out, float2 *vel_out, double *monitor, TickDuty duty, NextKeys nk,
             Members E) {
    pdl_enter();
    end_of_tick(duty, n_ptr);
    __shared__ __align__(128) float4 s_ps[SC_TILE_CAP];
    __shared__ __align__(128) float2 s_vel[SC_TILE_CAP];
    __shared__ __align__(128) uint2 s_pair[SC_K5_ROWS * SC_TILE];  // the block's first SC_K5_ROWS record slots
    __shared__ __align__(8) unsigned long long s_bar;
    const uint32_t b0 = blockIdx.x * SC_TILE;
    const uint32_t n = *n_ptr;
    if (b0 >= n) return;
    const uint32_t s = b0 + threadIdx.x;
    const bool live = s < n;
    const TileWindows w = tile_windows(desc + blockIdx.x);
    const uint32_t bar = smem_addr(&s_bar);
    const uint2 *my_rec = pair_rec + (size_t)blockIdx.x * (SC_MAX_NEIGHBORS * SC_TILE) + threadIdx.x;
    if (threadIdx.x == 0) mbar_init(bar, 1u);
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, (w.staged ? w.total * 24u : 0u) + SC_K5_ROWS * SC_TILE * 8u);
        bulk_g2s(smem_addr(s_pair), my_rec, SC_K5_ROWS * SC_TILE * 8u, bar);
        if (w.staged) {
            stage_windows(w, ps_in, 16u, smem_addr(s_ps), bar);
            stage_windows(w, vel, 8u, smem_addr(s_vel), bar);
        }
    }
    // everything this thread needs of its OWN particle, straight from global memory while the copies fly (the block is
    // a chain of latencies - descriptor, copies, these loads - and occupancy is set by shared memory, not registers:
    // nothing is gained by loading late)
    PS<float> me;
    int K = 0;
    double2 ps_own = make_double2(0, 0);
    float2 v_own = make_float2(0, 0);
    bool touching = false;
    uint32_t u = 0u;
    if (live) {
        if constexpr (kEns) u = E.uid[s];
        me = ps_in[s];
        K = pair_cnt[s];
        ps_own = pos[s];
        v_own = vel[s];
        touching = (wall_bits[s >> 5] >> (s & 31)) & 1u;
    }
    mbar_wait(bar, 0u);
    if (!live) return;
    DevParams Pm;
    if constexpr (kEns) Pm = member_params(E, u);
    const DevParams &P = pick_params<kEns>(P0, Pm);
    const float p_i = me.p;
    const float smooth = P.f_smooth, two_target = P.f_two_target;
    float tx = 0, ty = 0;         // F3 sum
    float qx = 0, qy = 0;         // F5 sum
    float sum_vx = 0, sum_vy = 0;  // sum of neighbor velocities (F6)
    const SmemAcc<float4> Aps{smem_addr_pinned(s_ps)};
    const SmemAcc<float2> Avel{smem_addr_pinned(s_vel)};
    const SmemAcc<uint2> Arec{smem_addr_pinned(s_pair) + threadIdx.x * 8u};
    // one pair: F3 pass 2 (crate.py:347-353), F5 (301-306), F6's neighbor velocity sum (319-323), in list order
    auto pair = [&](uint2 r, auto get_ps, auto get_vel) {
        uint32_t L;
        float nx, ny;
        pair_decode(r, L, nx, ny);
        const float4 nb = get_ps(L);
        const float2 vj = get_vel(L);
        const float ddx = me.sx - nb.y, ddy = me.sy - nb.z;
        const float align = (ddx * nx + ddy * ny) * smooth;
        const float fix = nb.x + p_i - two_target;
        const float cc = align + fix;
        const float ex = cc * nx, ey = cc * ny;
        const float ps_ = p_i + nb.x;
        const float fx = nx * ps_, fy = ny * ps_;
        // (the sums start at +0: in fp32 0 + x == x, so the reference's "first row assigns" needs no special case here -
        // unlike the fp64 kernel, where the bit pattern of -0 matters)
        tx += ex; ty += ey; qx += fx; qy += fy;
        sum_vx += vj.x; sum_vy += vj.y;
    };
    // the loop is unswitched on the two block-uniform / rare conditions: staged or pass-through block, and record slots
    // beyond the staged rows (K > SC_K5_ROWS: one particle in six at rest density), which come from global memory
    const int Ks = K < SC_K5_ROWS ? K : SC_K5_ROWS;
    if (w.staged) {
        auto gp = [&](uint32_t L) { return Aps.get(L); };
        auto gv = [&](uint32_t L) { return Avel.get(L); };
        for (int k = 0; k < Ks; ++k) pair(Arec.get((uint32_t)k * SC_TILE), gp, gv);
        for (int k = SC_K5_ROWS; k < K; ++k) pair(my_rec[k * SC_TILE], gp, gv);
    } else {
        auto gp = [&](uint32_t L) { const PS<float> g_ = ps_in[L]; return make_float4(g_.p, g_.sx, g_.sy, 0.0f); };
        auto gv = [&](uint32_t L) { return vel[L]; };
        for (int k = 0; k < Ks; ++k) pair(Arec.get((uint32_t)k * SC_TILE), gp, gv);
        for (int k = SC_K5_ROWS; k < K; ++k) pair(my_rec[k * SC_TILE], gp, gv);
    }
    force_tail<float, kMonitor, kEns>(s, K, p_i, tx, ty, qx, qy, P, W, ps_own, v_own, touching, wall_slot, wall_pre,
                                      pos_out, vel_out, monitor, n_ptr, nk, [&](float vx, float vy, float &ax, float &ay) {
        ax = sum_vx - (float)K * vx;
        ay = sum_vy - (float)K * vy;
    }, kEns ? member_of(E, u) * E.ncells : 0u);
}

// ------------------------------------------------------------------------------------------------------------
// Pair-record tap (sc_debug_pair_records): the records the last tick's density kernel left for the force kernel, as
// the force kernel reads them, in original index order.  One thread per sorted particle, blocks of SC_TILE, so that a
// block here is a block of the tiled kernels and its record region and windows are theirs.  Read-only on the step's
// buffers.  A record whose index does not map into the live set (which a correct run never writes) is reported as
// row -2 instead of being followed.
// `f64`: the fp64 kernels' records (index + vector arrays behind pair_off), else the tiled kernels' (sc_tile.cuh).
__global__ void __launch_bounds__(SC_TILE)
k_tap_pair_records(const uint32_t *n_ptr, bool f64, const BlockDesc *desc, const uint8_t *pair_cnt,
                   const uint32_t *pair_off, const uint32_t *pair_j, const void *pair_n, const uint32_t *uid,
                   const uint32_t *rank_of_uid, int *cnt_out, int *row_out, double2 *vec_out) {
    const uint32_t n = *n_ptr;
    const uint32_t s = blockIdx.x * SC_TILE + threadIdx.x;
    if (s >= n) return;
    const uint32_t r = rank_of_uid[uid[s]];
    const int K = pair_cnt[s];
    cnt_out[r] = K;
    TileWindows w{};
    if (!f64) w = tile_windows(desc + blockIdx.x);
    for (int k = 0; k < SC_MAX_NEIGHBORS; ++k) {
        const size_t o = (size_t)r * SC_MAX_NEIGHBORS + k;
        if (k >= K) { row_out[o] = -1; vec_out[o] = make_double2(0, 0); continue; }
        uint32_t j;
        double2 v;
        if (f64) {
            const size_t i = (size_t)pair_off[s] + k;
            j = pair_j[i];
            v = reinterpret_cast<const double2 *>(pair_n)[i];
        } else {
            const uint2 *rec = reinterpret_cast<const uint2 *>(pair_n);
            float nx, ny;
            pair_decode(rec[((size_t)blockIdx.x * SC_MAX_NEIGHBORS + k) * SC_TILE + threadIdx.x], j, nx, ny);
            v = make_double2((double)nx, (double)ny);
            if (w.staged) {  // local index in W0 | W1 | W2 -> sorted index
                uint32_t m = 0xFFFFFFFFu;
                for (int q = 0; q < 3; ++q)
                    if (j >= w.off[q] && j < w.off[q] + w.cnt[q]) m = w.base[q] + (j - w.off[q]);
                j = m;
            }
        }
        row_out[o] = j < n ? (int)rank_of_uid[uid[j]] : -2;
        vec_out[o] = v;
    }
}

}  // namespace sc
