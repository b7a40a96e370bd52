// sc_api.cu - context, launch orchestration and the C ABI declared in include/sandcrate.h.
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo (see sand_crate_b200/build.py).
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "sc_dist.cuh"

using namespace sc;

static std::string g_create_error;

enum Slot {
    SLOT_CLEAR = 0, SLOT_PREPASS, SLOT_SCAN, SLOT_PLACE, SLOT_RANK_GATHER, SLOT_DENSITY, SLOT_FORCE, SLOT_COUNT,
    SLOT_RANKMAP, SLOT_IO, SLOT_END, SLOT_DIST_PACK
};
static const char *k_slot_names[SC_PROFILE_SLOTS] = {
    "clear", "prepass_wall_key", "scan", "place", "rank_gather", "density", "force_integrate", "count_neighbors",
    "rank_map", "io_scatter", "end_tick", "dist_pack", "", "", "", ""};
// NVTX range per launch, named after the section of the reference's tick the kernel replaces (the `debug_timer`
// sections of crate.py:97-124, utils/timer.py:10-48) so a timeline reads like the reference's own Timer overlay
static const char *k_slot_nvtx[SC_PROFILE_SLOTS] = {
    "begin tick (clear cell grid)", "Virtual Colliders (remove, walls, hard wall fix, cell keys)",
    "Collisions: cell scan", "Collisions: counting-sort placement", "Collisions: in-cell rank + gather",
    "Collisions + Colliders + Pressure + tension pass 1 (density kernel)",
    "tension, gravity, pressure, viscosity, wall_bounce, continuous_collision, integrate (force kernel)",
    "tap: neighbor counts", "readback: uid -> row map", "readback / upload", "end tick",
    "strips: pack", "", "", "", ""};

struct ProfEvent { int slot; cudaEvent_t e0, e1; };

struct sc_ctx {
    int device = 0, precision = 0;
    int64_t cap = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    sc_params hp{};
    bool params_set = false, walls_set = false;
    DevParams dp{};
    Grid grid{};
    WallParams walls{};
    int grid_contacts = 1;  // wall contacts per particle the cell grid has room for (world_rows); only ever grows
    int noise_mode = SC_NOISE_NONE;
    uint64_t seed = 0, tick = 0;
    // particle state: *_cur = current state (order left by the previous tick), *_srt = this tick's sorted gather
    double2 *pos_cur = nullptr, *pos_srt = nullptr;
    float2 *rel_srt = nullptr;        // cell-relative fp32 positions of the sorted set
    float4 *rec_srt = nullptr;        // mixed mode: (rel, cell column, uid) search records of the tiled pair kernels
    BlockDesc *blk_desc = nullptr;    // mixed mode: per block of SC_TILE sorted particles, its three windows
    void *vel_cur = nullptr, *vel_srt = nullptr;
    uint32_t *uid_cur = nullptr, *uid_srt = nullptr;
    uint32_t *cell_key = nullptr, *cell_key_srt = nullptr, *tmpidx = nullptr;
    // One cell-count grid and one cell_start array (+ the live count at [ncells]).  The counts are zero between ticks:
    // k_place takes each one back down (sc_sort.cuh).  cell_start holds the last search's boundaries until the next
    // tick's scan (the taps and the strip pack read them).
    uint32_t *cell_count = nullptr, *cell_start = nullptr; size_t cell_cap = 0;
    // The wall bitmaps, side list and its counter are double buffered by tick parity: the force kernel of one tick may
    // fill the next tick's (NextKeys) while it reads its own.  wall_bits_* / wall_pre point at the last search's set.
    int par = 0;
    bool next_clean = false;  // the next tick finds the grid, its wall set and the scan descriptors cleared
    // The last force kernel ran the next tick's key pass (NextKeys, sc_pair.cuh) and nothing since changed what the keys
    // depend on: the next tick launches no k_prepass.  pos_cur then holds the positions AFTER the next tick's hard-wall
    // fix (the readback undoes it: k_scatter_pos), and drop_keys() takes it all back when a call invalidates it.
    bool next_keyed = false;
    bool keys_dropped = true;  // a call since the last step invalidated the keys: this step's force kernel computes none
    unsigned long long *bsum = nullptr; size_t bsum_cap = 0;    // cell scan: tile descriptors, [0] = ticket
    unsigned long long *bsum2 = nullptr; size_t bsum2_cap = 0;  // the same for every other scan (readback maps)
    void *ps = nullptr;               // PS<Real>[cap]: pressure + surface normal of the sorted set
    uint32_t *pair_j = nullptr; void *pair_n = nullptr;  // [cap * SC_MAX_NEIGHBORS], written by K4, read by K5
    uint32_t *pair_off = nullptr; uint8_t *pair_cnt = nullptr;
    uint32_t *wbits_cur[2] = {nullptr, nullptr}, *wbits_srt[2] = {nullptr, nullptr};
    uint32_t *wall_bits_cur = nullptr, *wall_bits_srt = nullptr, *wall_slot_cur = nullptr, *wall_slot_srt = nullptr;
    double2 *wall_pre_buf[2] = {nullptr, nullptr}, *wall_pre = nullptr;
    Counters *cnt = nullptr;
    uint32_t *rank_of_uid = nullptr; size_t uid_cap = 0;
    uint32_t next_uid = 0;
    uint32_t *count_by_rank = nullptr, *list_sorted = nullptr;
    double *noise_dev = nullptr; size_t noise_cap = 0;
    double2 *stage2 = nullptr; double *stage1 = nullptr;
    int64_t n_host = 0;       // upper bound on the live count; exact when n_exact
    bool n_exact = true;
    bool in_step = false;     // between sc_step_begin and sc_step_finish
    bool srt_valid = false;   // *_srt arrays hold the last tick's search state
    bool rows_valid = false;  // pos_cur / uid_cur are still in the order of the last search (cell rows ascending)
    bool lists_valid = false, rank_valid = false;
    bool carry_count = false; // the device count must be refreshed from the previous tick's scan total
    bool monitor_on = false;  // ForceMonitor mode: K5 also sums |dv| per force stage
    double *monitor = nullptr; // 6 sums + particle count of the last tick
    bool dist_on = false;     // strip decomposition: particle arrays hold owned + ghost particles
    DistCfg dist{};
    // [0], [1]: send headers standing in for a missing lower / upper neighbor's; [2].count: the "blocks done"
    // counter of the direct pack kernel (k_dist_pack<..., true>)
    WireHeader *wire_dummy = nullptr;
    WireHeader *send_lo = nullptr, *send_hi = nullptr;  // the send buffers of the last pack (re-armed by the pre-pass)
    // The unpack waits for the neighbors' records, and nothing of the tick's first pass over the particles this rank
    // already holds (walls, cell keys) depends on them: the unpack is therefore DEFERRED - recorded here by
    // sc_dist_unpack[_flagged] and carried out by the step's pre-pass itself (PrepassUnpack), whose blocks behind the
    // particles already held wait for the flags and read the receive buffers directly.  One launch less on the critical
    // path; the neighbors' latency hides behind the pass over the resident particles.  Until that step, the particle
    // arrays and the device count lack the records: enter() refuses every call that would read or change them.
    struct { bool on = false; const void *recv_lo = nullptr, *flag_lo = nullptr, *recv_hi = nullptr, *flag_hi = nullptr;
             uint32_t value = 0; } pend;
    int64_t launches = 0;
    int64_t syncs = 0;        // host waits on the stream (cudaStreamSynchronize) issued by this context's entry points
    bool profiling = false;
    std::vector<ProfEvent> pending;
    std::vector<cudaEvent_t> pool;
    int64_t prof_launches[SC_PROFILE_SLOTS] = {0};
    double prof_ms[SC_PROFILE_SLOTS] = {0};
};

__global__ void k_end_tick(Counters *cnt, const uint32_t *total) { cnt->n = *total; }

static int fail(sc_ctx *c, const std::string &m) {
    if (c) c->err = m; else g_create_error = m;
    return 1;
}
static cudaError_t stream_sync(sc_ctx *c) { c->syncs++; return cudaStreamSynchronize(c->stream); }
#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return fail(ctx, std::string(#call) + ": " + cudaGetErrorString(e_) + " (" __FILE__ ":" +   \
                                 std::to_string(__LINE__) + ")");                                       \
    } while (0)
#define CKR(expr)            \
    do {                     \
        int r_ = (expr);     \
        if (r_) return r_;   \
    } while (0)

// Prologue of the entry points that take a context.  Between sc_dist_unpack[_flagged] and the step that carries the
// unpack out, only the calls that consume it (`consumes_unpack`: sc_step, sc_step_n, sc_step_begin) pass.  The calls
// that never touch the particle state (sc_set_tick, sc_synchronize, sc_destroy, sc_last_error, measurement) skip it.
static int enter(sc_ctx *ctx, const char *who, bool consumes_unpack = false) {
    if (!ctx) return fail(ctx, std::string(who) + ": NULL ctx");
    if (ctx->pend.on && !consumes_unpack)
        return fail(ctx, std::string(who) + ": a strip unpack is pending (the next call must be a step)");
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return fail(ctx, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    return 0;
}

// launch with programmatic stream serialization (see pdl_enter in sc_common.cuh)
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

static inline unsigned blocks_for(int64_t n) { return (unsigned)((n + SC_BLOCK - 1) / SC_BLOCK); }

struct ProfScope {
    sc_ctx *c; int slot; cudaEvent_t e0 = nullptr, e1 = nullptr;
    ProfScope(sc_ctx *c_, int slot_) : c(c_), slot(slot_) {
        c->launches++;
        nvtxRangePushA(k_slot_nvtx[slot]);  // a no-op unless a profiler has injected itself
        if (!c->profiling) return;
        auto get = [&]() {
            cudaEvent_t e;
            if (!c->pool.empty()) { e = c->pool.back(); c->pool.pop_back(); } else cudaEventCreate(&e);
            return e;
        };
        e0 = get(); e1 = get();
        cudaEventRecord(e0, c->stream);
    }
    ~ProfScope() {
        nvtxRangePop();
        if (!c->profiling) return;
        cudaEventRecord(e1, c->stream);
        c->pending.push_back({slot, e0, e1});
    }
};

static int prof_flush(sc_ctx *ctx) {
    if (ctx->pending.empty()) return 0;
    CK(stream_sync(ctx));
    for (auto &p : ctx->pending) {
        float ms = 0;
        cudaEventElapsedTime(&ms, p.e0, p.e1);
        ctx->prof_ms[p.slot] += ms;
        ctx->prof_launches[p.slot]++;
        ctx->pool.push_back(p.e0);
        ctx->pool.push_back(p.e1);
    }
    ctx->pending.clear();
    return 0;
}

// SC_POISON=<byte> (developer switch): fill every allocation with that byte, so that a read of memory nothing has
// written shows up as garbage (0xFF: NaN / invalid index) instead of whatever a recycled allocation happened to hold
static int poison_byte() {
    static int b = -2;
    if (b == -2) { const char *e = getenv("SC_POISON"); b = e ? (int)strtol(e, nullptr, 0) & 0xFF : -1; }
    return b;
}
template <typename T> static int dev_alloc(sc_ctx *ctx, T **p, size_t count) {
    CK(cudaMalloc((void **)p, sizeof(T) * (count ? count : 1)));
    if (poison_byte() >= 0) {
        CK(cudaMemset((void *)*p, poison_byte(), sizeof(T) * (count ? count : 1)));
        CK(cudaDeviceSynchronize());  // the fill runs on the legacy stream; the context's stream does not wait for it
    }
    return 0;
}
static size_t real_size(const sc_ctx *c) { return c->precision == SC_PRECISION_F64 ? 8 : 4; }

// ---------------------------------------------------------------------------------------------------------
static int setup_grid(sc_ctx *ctx, double d, int row_min, int row_max, int col_min, int col_max) {
    // one margin cell on every side so the 3x3 neighborhood never leaves the array
    Grid g;
    g.d = d;
    g.inv_d = 1.0 / d;
    g.row_min = row_min - 1;
    g.col_min = col_min - 1;
    const int64_t nrows = (int64_t)row_max - row_min + 3, ncols = (int64_t)col_max - col_min + 3;
    if (nrows <= 0 || ncols <= 0 || nrows * ncols > (int64_t)1 << 31)
        return fail(ctx, "cell grid too large: " + std::to_string(nrows) + " x " + std::to_string(ncols));
    g.nrows = (int)nrows;
    g.ncols = (int)ncols;
    g.ncells = (uint32_t)(nrows * ncols);
    const size_t need = (size_t)g.ncells + 8;  // + the live count at [ncells]; bulk copies read whole 16-byte groups
    if (need > ctx->cell_cap) {
        if (ctx->cell_count) CK(cudaFree(ctx->cell_count));
        if (ctx->cell_start) CK(cudaFree(ctx->cell_start));
        CKR(dev_alloc(ctx, &ctx->cell_count, need));
        CKR(dev_alloc(ctx, &ctx->cell_start, need));
        ctx->cell_cap = need;
    }
    ctx->next_clean = false;  // a new grid: the next tick clears it itself
    ctx->next_keyed = false;  // (every caller has dropped the keys first: drop_keys)
    const size_t nb = (size_t)(g.ncells + SC_SCAN_TILE - 1) / SC_SCAN_TILE + 2;
    const size_t nb2 = (size_t)(ctx->cap + SC_SCAN_TILE - 1) / SC_SCAN_TILE + 2;
    const size_t needb = nb > nb2 ? nb : nb2;
    if (needb > ctx->bsum_cap) {
        if (ctx->bsum) CK(cudaFree(ctx->bsum));
        CKR(dev_alloc(ctx, &ctx->bsum, needb));
        ctx->bsum_cap = needb;
    }
    ctx->grid = g;
    return 0;
}

static void refresh_wall_boxes(sc_ctx *ctx);
static int contact_bound(const WallParams &w);
static int sync_count(sc_ctx *ctx);
static void refresh_count(sc_ctx *ctx);

#define SC_DIST_ROW_SLACK 96
#define SC_K5_THREADS 128  // K5 block size: 128 measured 2 us faster than 256 (blocks drain sooner, the gather-latency-bound kernel keeps more warps resident)

// Rows (= columns) of the world box's cell grid.  Live particles satisfy -r <= coord <= 1 + r (crate.py:152) before
// apply_hard_wall_fix, which adds one push of r - dist <= r per wall contact: with V contacts a particle moves by up to
// V r.  The grid has room for grid_contacts contacts, so every position the search sees lies in an interior cell (a
// clamped one would merge rows the reference keeps apart).  With one contact this is the grid of a contact-free scene.
static void world_rows(const sc_ctx *ctx, long long &lo, long long &hi) {
    const double d = ctx->dp.d, r = ctx->dp.r, m = r + ctx->grid_contacts * r;
    lo = (long long)std::floor(-m / d) - 1;
    hi = (long long)std::floor((1 + m) / d) + 1;
}

// Cell grid of the world box; in strip mode only the rows this rank can ever hold (its strip, the halo, and the
// one-row shift the wall fix can add), so clearing and scanning the grid scales with the strip, not the scene.
static int world_grid(sc_ctx *ctx) {
    long long wlo, whi;
    world_rows(ctx, wlo, whi);
    if (wlo < -(1LL << 30) || whi > (1LL << 30)) return fail(ctx, "cell grid too large for the wall-fix margin");
    const int lo = (int)wlo, hi = (int)whi;
    int rlo = lo, rhi = hi;
    if (ctx->dist_on) {
        // halo + wall-fix shift + slack for cuts that slide while the partition is re-balanced (sc_dist_set_rows)
        const long long margin = ctx->dist.halo + 2 + SC_DIST_ROW_SLACK;
        if (ctx->dist.has_lo && ctx->dist.row_lo - margin > rlo) rlo = (int)(ctx->dist.row_lo - margin);
        if (ctx->dist.has_hi && ctx->dist.row_hi + margin < rhi) rhi = (int)(ctx->dist.row_hi + margin);
    }
    CKR(setup_grid(ctx, ctx->dp.d, rlo, rhi, lo, hi));
    ctx->srt_valid = false; ctx->rows_valid = false;
    return 0;
}

static int refresh_dev_params(sc_ctx *ctx) {
    const sc_params &h = ctx->hp;
    DevParams &p = ctx->dp;
    p.dt = h.dt; p.r = h.particle_radius; p.d = h.particle_radius * 2;  // crate.py:65-67
    p.touch = h.particle_radius * 1.2;                                   // crate.py:229
    p.decay = h.wall_collision_decay; p.amp = h.pressure_amplifier; p.ignored = h.ignored_pressure;
    p.level = h.collider_noise_level; p.visc = h.viscosity; p.smooth = h.surface_smoothing;
    p.target = h.target_pressure; p.gx = h.gravity_x; p.gy = h.gravity_y;
    p.box_lo = -h.particle_radius; p.box_hi = 1 + h.particle_radius;     // crate.py:152
    // fp32 constants of the mixed-precision kernels: the same operations, in the same order, the kernels used per thread
    p.f_d = (float)p.d; p.f_inv_d = (float)(1.0 / p.d); p.f_amp = (float)(p.d * p.level);
    p.f_band_hi = (p.f_d * p.f_d) * (1.0f + 4e-6f); p.f_band_lo = (p.f_d * p.f_d) * (1.0f - 4e-6f);
    p.f_dt = (float)p.dt; p.f_dt_gx = (float)(p.dt * p.gx); p.f_dt_gy = (float)(p.dt * p.gy);
    p.f_dt_amp = (float)(p.dt * p.amp); p.f_dt_visc = (float)(p.dt * p.visc);
    p.f_smooth = (float)p.smooth; p.f_two_target = (float)(2 * p.target); p.f_ignored = (float)p.ignored;
    return 0;
}

// k_begin_tick over the cell-count grid and the wall set of tick parity `q` (see there for `carry` and `restore`)
static int launch_clear(sc_ctx *ctx, int q, const uint32_t *carry, KeyRestore restore) {
    const Grid &g = ctx->grid;
    ProfScope ps(ctx, SLOT_CLEAR);
    const uint32_t words = (uint32_t)(ctx->cap / 32 + 1);
    const unsigned nb = (unsigned)std::min<int64_t>(((int64_t)g.ncells / 4 + SC_BLOCK - 1) / SC_BLOCK + 1, 148 * 16);
    const uint32_t scan_words = (g.ncells + SC_SCAN_TILE - 1) / SC_SCAN_TILE + 1;  // ticket + descriptors
    CK(launch_pdl(k_begin_tick, dim3(nb), dim3(SC_BLOCK), ctx->stream, ctx->cnt, ctx->cell_count, g.ncells, carry,
                  ctx->wbits_cur[q], ctx->wbits_srt[q], words, ctx->bsum, scan_words, (uint32_t)ctx->cap, restore));
    return 0;
}

// Called by every entry point that changes what the next tick's keys depend on - the particle state and count, the
// walls, the parameters, the cell grid, the strip exchange - before it changes anything.  If the last force kernel
// already ran the next tick's key pass (next_keyed), its work is taken back: positions from before its hard-wall fix,
// counts and the next tick's wall set zeroed (one launch).  The next tick then runs its own pre-pass, and its force
// kernel computes no keys for the tick after (keys_dropped): a scene that changes its walls every tick (a moving
// paddle) would otherwise pay for keys and their clearing every tick only to throw them away.
static int drop_keys(sc_ctx *ctx) {
    ctx->keys_dropped = true;
    if (!ctx->next_keyed) return 0;
    ctx->next_keyed = false;
    const int q = ctx->par ^ 1;
    CKR(launch_clear(ctx, q, nullptr, KeyRestore{ctx->pos_cur, ctx->wall_slot_cur, ctx->wall_pre_buf[q]}));
    ctx->next_clean = true;
    return 0;
}

extern "C" int sc_version(void) { return 1; }

extern "C" const char *sc_last_error(const sc_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int sc_create(int device, int precision, int64_t capacity, void *stream, sc_ctx **out) {
    sc_ctx *ctx = nullptr;
    if (!out) return fail(nullptr, "sc_create: out is NULL");
    *out = nullptr;
    if (precision != SC_PRECISION_F64 && precision != SC_PRECISION_MIXED) return fail(nullptr, "sc_create: bad precision");
    if (capacity < 1 || capacity > (int64_t)SC_IDX_MASK) return fail(nullptr, "sc_create: capacity out of range");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, std::string("sc_create: no CUDA device (") + cudaGetErrorString(e) +
                                 "); this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, "sc_create: bad device index");
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major != 10)
        return fail(nullptr, "sc_create: device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                                 ", this build targets sm_100a only");
    sc_ctx *c = new sc_ctx();
    ctx = c;
    c->device = device; c->precision = precision; c->cap = capacity;
    if (stream) c->stream = (cudaStream_t)stream;
    else { cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking); c->own_stream = true; }
    // + 16: the tiled kernels bulk-copy windows whose ends are rounded up to 16-byte groups
    const size_t n = (size_t)capacity + 16, rs = real_size(c);
    int rc = 0;
    rc |= dev_alloc(c, &c->pos_cur, n); rc |= dev_alloc(c, &c->pos_srt, n);
    rc |= dev_alloc(c, (char **)&c->vel_cur, n * 2 * rs); rc |= dev_alloc(c, (char **)&c->vel_srt, n * 2 * rs);
    rc |= dev_alloc(c, &c->uid_cur, n); rc |= dev_alloc(c, &c->uid_srt, n);
    rc |= dev_alloc(c, &c->cell_key, n); rc |= dev_alloc(c, &c->cell_key_srt, n);
    rc |= dev_alloc(c, &c->tmpidx, n);
    rc |= dev_alloc(c, &c->rel_srt, n);
    if (precision == SC_PRECISION_MIXED) {
        rc |= dev_alloc(c, &c->rec_srt, n);
        rc |= dev_alloc(c, &c->blk_desc, (n + SC_TILE - 1) / SC_TILE + 1);
    }
    rc |= dev_alloc(c, (char **)&c->ps, n * 4 * rs);
    // pair records: the fp64 kernels bump-allocate (pair_off); the tiled kernels give every block of SC_TILE sorted
    // particles its own slot-major region of SC_TILE x 20 records, so the buffer holds whole blocks
    const size_t npair = ((n + SC_TILE - 1) / SC_TILE) * SC_TILE * SC_MAX_NEIGHBORS;
    rc |= dev_alloc(c, &c->pair_j, precision == SC_PRECISION_F64 ? npair : 1);
    rc |= dev_alloc(c, (char **)&c->pair_n, npair * 2 * rs);
    if (!rc) cudaMemsetAsync(c->pair_n, 0, npair * 2 * rs, c->stream);  // K5 bulk-copies slots K4 may not have written
    rc |= dev_alloc(c, &c->pair_off, precision == SC_PRECISION_F64 ? n : 1);
    rc |= dev_alloc(c, &c->pair_cnt, n);
    for (int q = 0; q < 2; ++q) { rc |= dev_alloc(c, &c->wbits_cur[q], n / 32 + 1); rc |= dev_alloc(c, &c->wbits_srt[q], n / 32 + 1); }
    c->wall_bits_cur = c->wbits_cur[0]; c->wall_bits_srt = c->wbits_srt[0];
    rc |= dev_alloc(c, &c->wall_slot_cur, n); rc |= dev_alloc(c, &c->wall_slot_srt, n);
    rc |= dev_alloc(c, &c->wall_pre_buf[0], n); rc |= dev_alloc(c, &c->wall_pre_buf[1], n);
    c->wall_pre = c->wall_pre_buf[0];
    rc |= dev_alloc(c, &c->cnt, 1);
    rc |= dev_alloc(c, &c->count_by_rank, n + 1);
    rc |= dev_alloc(c, &c->stage2, n); rc |= dev_alloc(c, &c->stage1, n);
    if (rc) { g_create_error = c->err; sc_destroy(c); return 1; }
    cudaMemsetAsync(c->cnt, 0, sizeof(Counters), c->stream);
    c->walls.S = 0; c->walls.nbodies = 0;
    *out = c;
    return 0;
}

extern "C" void sc_destroy(sc_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    void *ptrs[] = {c->pos_cur, c->pos_srt, c->vel_cur, c->vel_srt, c->uid_cur, c->uid_srt, c->cell_key,
                    c->cell_key_srt, c->tmpidx, c->cell_count, c->cell_start, c->bsum, c->bsum2, c->rel_srt, c->rec_srt, c->blk_desc, c->ps, c->pair_j, c->pair_n, c->pair_off, c->pair_cnt,
                    c->wbits_cur[0], c->wbits_cur[1], c->wbits_srt[0], c->wbits_srt[1], c->wall_slot_cur, c->wall_slot_srt, c->wall_pre_buf[0], c->wall_pre_buf[1], c->cnt,
                    c->rank_of_uid, c->count_by_rank, c->list_sorted, c->noise_dev, c->stage2, c->stage1, c->wire_dummy, c->monitor};
    for (void *p : ptrs) if (p) cudaFree(p);
    for (auto &p : c->pending) { cudaEventDestroy(p.e0); cudaEventDestroy(p.e1); }
    for (auto e : c->pool) cudaEventDestroy(e);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int sc_set_params(sc_ctx *ctx, const sc_params *p) {
    CKR(enter(ctx, "sc_set_params"));
    if (!p) return fail(ctx, "sc_set_params: NULL argument");
    if (!(p->particle_radius > 0) || !(p->dt == p->dt)) return fail(ctx, "sc_set_params: particle_radius must be > 0");
    const bool regrid = !ctx->params_set || p->particle_radius != ctx->hp.particle_radius;
    if (regrid && ctx->in_step) return fail(ctx, "sc_set_params: radius change inside a split step");
    // the same bytes again (a Crate pushes its coefficients every tick) leave the next tick's keys valid
    if (!ctx->params_set || std::memcmp(p, &ctx->hp, sizeof(sc_params)) != 0) CKR(drop_keys(ctx));
    if (regrid && ctx->params_set) CKR(sync_count(ctx));  // the live count sits in the old cell array's tail
    ctx->hp = *p;
    refresh_dev_params(ctx);
    if (regrid) {
        if (ctx->walls_set) {
            sc_pad_segments(&ctx->walls.seg[0][0], ctx->walls.S, ctx->dp.r, &ctx->walls.pad[0][0]);
            refresh_wall_boxes(ctx);
            ctx->grid_contacts = std::max(ctx->grid_contacts, contact_bound(ctx->walls));
        }
        CKR(world_grid(ctx));  // room for the wall fix's shift (world_rows)
    }
    ctx->params_set = true;
    return 0;
}

extern "C" int sc_pad_segments(const double *segments, int S, double pad, double *padded) {
    // geometry_utils.py:146-172.  Host code of this file is built with -ffp-contract=off.
    for (int k = 0; k < S; ++k) {
        const double ax = segments[4 * k], ay = segments[4 * k + 1], bx = segments[4 * k + 2], by = segments[4 * k + 3];
        const double abx = bx - ax, aby = by - ay;
        const double nx = aby, ny = -abx;
        const double norm = std::sqrt(nx * nx + ny * ny);
        const double ox = nx * pad / norm, oy = ny * pad / norm;
        double *p1 = padded + 4 * k, *p2 = padded + 4 * (S + k);
        p1[0] = ax + ox; p1[1] = ay + oy; p1[2] = bx + ox; p1[3] = by + oy;
        p2[0] = bx - ox; p2[1] = by - oy; p2[2] = ax - ox; p2[3] = ay - oy;
    }
    return 0;
}

// bounding boxes for the conservative culls of WallParams (grown so that rounding can never cull a true hit)
static void refresh_wall_boxes(sc_ctx *ctx) {
    WallParams &w = ctx->walls;
    auto grow = [](double *box, double ax, double ay, double bx, double by, double m) {
        const double xmin = std::fmin(ax, bx), xmax = std::fmax(ax, bx), ymin = std::fmin(ay, by), ymax = std::fmax(ay, by);
        const double scale = std::fmax(1.0, std::fmax(std::fmax(std::fabs(xmin), std::fabs(xmax)),
                                                      std::fmax(std::fabs(ymin), std::fabs(ymax))));
        const double e = m * (1.0 + 1e-6) + 1e-12 * scale;
        box[0] = xmin - e; box[1] = xmax + e; box[2] = ymin - e; box[3] = ymax + e;
    };
    for (int k = 0; k < w.S; ++k) grow(w.seg_box[k], w.seg[k][0], w.seg[k][1], w.seg[k][2], w.seg[k][3], ctx->dp.touch);
    for (int k = 0; k < 2 * w.S; ++k) grow(w.pad_box[k], w.pad[k][0], w.pad[k][1], w.pad[k][2], w.pad[k][3], 0.0);
    // Largest-area-greedy rectangle inside the world box that meets none of the boxes.  Only ever used as
    // "strictly inside -> nothing to test", so any rectangle that meets no box is correct; greedy just makes it big.
    auto safe_rect = [&](double (*boxes)[4], int nb, double *out) {
        double r[4] = {ctx->dp.box_lo, ctx->dp.box_hi, ctx->dp.box_lo, ctx->dp.box_hi};
        auto meets = [&](const double *b) { return b[0] < r[1] && b[1] > r[0] && b[2] < r[3] && b[3] > r[2]; };
        for (int pass = 0; pass < nb + 1; ++pass) {
            bool changed = false;
            for (int k = 0; k < nb; ++k) {
                const double *b = boxes[k];
                if (!meets(b)) continue;
                const double w_ = r[1] - r[0], h_ = r[3] - r[2];
                const double area[4] = {(r[1] - b[1]) * h_, (b[0] - r[0]) * h_, w_ * (r[3] - b[3]), w_ * (b[2] - r[2])};
                int best = 0;
                for (int q = 1; q < 4; ++q) if (area[q] > area[best]) best = q;
                if (best == 0) r[0] = b[1]; else if (best == 1) r[1] = b[0]; else if (best == 2) r[2] = b[3]; else r[3] = b[2];
                changed = true;
            }
            if (!changed) break;
        }
        bool ok = r[0] < r[1] && r[2] < r[3];
        for (int k = 0; ok && k < nb; ++k) ok = !meets(boxes[k]);
        if (!ok) { r[0] = 1; r[1] = 0; r[2] = 1; r[3] = 0; }  // empty: nothing is skipped
        for (int q = 0; q < 4; ++q) out[q] = r[q];
    };
    safe_rect(w.seg_box, w.S, w.safe_contact);
    safe_rect(w.pad_box, 2 * w.S, w.safe_ccd);
    // fp32 copy, shrunk by far more than the fp32 rounding of a coordinate in [-1, 2] (6e-8) and of a movement
    if (w.safe_ccd[0] < w.safe_ccd[1]) {
        w.safe_ccd_f32[0] = (float)(w.safe_ccd[0] + 1e-6); w.safe_ccd_f32[1] = (float)(w.safe_ccd[1] - 1e-6);
        w.safe_ccd_f32[2] = (float)(w.safe_ccd[2] + 1e-6); w.safe_ccd_f32[3] = (float)(w.safe_ccd[3] - 1e-6);
    } else {
        w.safe_ccd_f32[0] = 1.0f; w.safe_ccd_f32[1] = 0.0f; w.safe_ccd_f32[2] = 1.0f; w.safe_ccd_f32[3] = 0.0f;
    }
}

// The most wall contacts one particle can have: the largest number of touch boxes (seg_box) that share a point.  A
// contact needs the particle inside its segment's box (the cull of key_particle), so no particle has more.  The deepest
// point of a set of closed boxes is the lower-left corner of their intersection, (xmin of one box, ymin of another):
// trying those S^2 points is exact.  At least 1, so a grid is never smaller than a one-contact grid.
static int contact_bound(const WallParams &w) {
    int best = 1;
    for (int i = 0; i < w.S; ++i)
        for (int j = 0; j < w.S; ++j) {
            const double x = w.seg_box[i][0], y = w.seg_box[j][2];
            int n = 0;
            for (int k = 0; k < w.S; ++k)
                n += x >= w.seg_box[k][0] && x <= w.seg_box[k][1] && y >= w.seg_box[k][2] && y <= w.seg_box[k][3];
            best = std::max(best, n);
        }
    return best;
}

extern "C" int sc_set_walls(sc_ctx *ctx, const double *segments, int S, const int32_t *body_len,
                            const double *body_kin, int nbodies) {
    CKR(enter(ctx, "sc_set_walls"));
    if (S < 0 || S > SC_MAX_SEGMENTS) return fail(ctx, "sc_set_walls: more than SC_MAX_SEGMENTS segments");
    if (nbodies < 0 || nbodies > SC_MAX_BODIES) return fail(ctx, "sc_set_walls: more than SC_MAX_BODIES bodies");
    if (!ctx->params_set) return fail(ctx, "sc_set_walls: call sc_set_params first (padding needs the radius)");
    WallParams &w = ctx->walls;
    {   // the same walls again (a Crate pushes them every tick) leave the next tick's keys valid; moving ones do not
        bool same = ctx->walls_set && S == w.S && nbodies == w.nbodies &&
                    (S == 0 || std::memcmp(&w.seg[0][0], segments, sizeof(double) * 4 * (size_t)S) == 0);
        int k = 0;
        for (int b = 0; same && b < nbodies; ++b) {
            same = std::memcmp(w.kin[b], body_kin + 5 * b, sizeof(double) * 5) == 0;
            for (int q = 0; same && q < body_len[b]; ++q, ++k) same = k < S && w.seg_body[k] == b;
        }
        if (!same || k != S) CKR(drop_keys(ctx));
    }
    w.S = S; w.nbodies = nbodies;
    int k = 0;
    for (int b = 0; b < nbodies; ++b) {
        for (int q = 0; q < body_len[b]; ++q) {
            if (k >= S) return fail(ctx, "sc_set_walls: body_len does not sum to S");
            w.seg_body[k++] = b;
        }
        for (int q = 0; q < 5; ++q) w.kin[b][q] = body_kin[5 * b + q];
    }
    if (k != S) return fail(ctx, "sc_set_walls: body_len does not sum to S");
    if (S) std::memcpy(&w.seg[0][0], segments, sizeof(double) * 4 * (size_t)S);
    sc_pad_segments(&w.seg[0][0], S, ctx->dp.r, &w.pad[0][0]);
    refresh_wall_boxes(ctx);
    ctx->walls_set = true;
    // walls that can give a particle more contacts than the grid has room for: a larger grid (never a smaller one, so
    // a moving body does not re-grid back and forth).  refresh_count carries the live count out of the old cell
    // array on the stream: no host wait.
    const int v = contact_bound(w);
    if (v > ctx->grid_contacts) {
        if (ctx->in_step) return fail(ctx, "sc_set_walls: walls that need a larger cell grid inside a split step");
        CKR(drop_keys(ctx));
        refresh_count(ctx);
        ctx->grid_contacts = v;
        CKR(world_grid(ctx));
    }
    return 0;
}

extern "C" int sc_set_noise(sc_ctx *ctx, int mode, uint64_t seed) {
    CKR(enter(ctx, "sc_set_noise"));
    if (mode < SC_NOISE_NONE || mode > SC_NOISE_HOST) return fail(ctx, "sc_set_noise: bad mode");
    ctx->noise_mode = mode; ctx->seed = seed;
    return 0;
}
extern "C" int sc_set_tick(sc_ctx *ctx, uint64_t tick) {
    if (!ctx) return fail(ctx, "sc_set_tick: NULL ctx");
    ctx->tick = tick;
    return 0;
}

// a step ran since cnt->n was last written (no force kernel carried the count): its scan total is the live count
static void refresh_count(sc_ctx *ctx) {
    if (!ctx->carry_count) return;
    ProfScope ps(ctx, SLOT_END);
    k_end_tick<<<1, 1, 0, ctx->stream>>>(ctx->cnt, ctx->cell_start + ctx->grid.ncells);
    ctx->carry_count = false;
}

static int sync_count(sc_ctx *ctx) {
    refresh_count(ctx);
    if (ctx->n_exact) return 0;
    Counters h;
    CK(cudaMemcpyAsync(&h, ctx->cnt, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    ctx->n_host = h.n;
    ctx->n_exact = true;
    return 0;
}

static int upload_particles(sc_ctx *ctx, const double *pos, const double *vel, int64_t at, int64_t n) {
    if (n == 0) return 0;
    // bit 31 of a uid marks a ghost copy (sc_dist.cuh) and the uid -> row map grows with every particle ever created
    if ((uint64_t)ctx->next_uid + (uint64_t)n >= (uint64_t)SC_GHOST_BIT)
        return fail(ctx, "particle identities exhausted (2^31 particles created in this context)");
    CK(cudaMemcpyAsync(ctx->pos_cur + at, pos, sizeof(double2) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->precision == SC_PRECISION_F64) {
        CK(cudaMemcpyAsync((double2 *)ctx->vel_cur + at, vel, sizeof(double2) * (size_t)n, cudaMemcpyHostToDevice,
                           ctx->stream));
    } else {
        CK(cudaMemcpyAsync(ctx->stage2, vel, sizeof(double2) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        ProfScope ps(ctx, SLOT_IO);
        k_convert_vel_in<float><<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(ctx->stage2, (float2 *)ctx->vel_cur + at,
                                                                            (uint32_t)n);
    }
    {
        ProfScope ps(ctx, SLOT_IO);
        k_iota<<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(ctx->uid_cur + at, ctx->next_uid, (uint32_t)n);
    }
    ctx->next_uid += (uint32_t)n;
    const uint32_t newn = (uint32_t)(at + n);
    CK(cudaMemcpyAsync(&ctx->cnt->n, &newn, sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    CK(stream_sync(ctx));  // host buffers are borrowed for the duration of the call only
    ctx->n_host = at + n;
    ctx->n_exact = true;
    ctx->rank_valid = false;
    return 0;
}

extern "C" int sc_set_state(sc_ctx *ctx, const double *pos, const double *vel, int64_t n) {
    CKR(enter(ctx, "sc_set_state"));
    CKR(drop_keys(ctx));
    if (n < 0 || n > ctx->cap) return fail(ctx, "sc_set_state: n exceeds capacity");
    if (ctx->in_step) return fail(ctx, "sc_set_state: inside a split step");
    ctx->next_uid = 0;
    ctx->srt_valid = false; ctx->lists_valid = false; ctx->rows_valid = false;
    ctx->carry_count = false;  // the count is (re)defined by the host below
    const uint32_t zero = 0;
    CK(cudaMemcpyAsync(&ctx->cnt->n, &zero, sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    ctx->n_host = 0; ctx->n_exact = true;
    return upload_particles(ctx, pos, vel, 0, n);
}

extern "C" int sc_set_state_uids(sc_ctx *ctx, const double *pos, const double *vel, const uint32_t *uid, int64_t n) {
    CKR(enter(ctx, "sc_set_state_uids"));
    if (!uid) return fail(ctx, "sc_set_state_uids: uid is NULL");
    uint32_t top = 0;
    for (int64_t i = 0; i < n; ++i) {
        if (uid[i] & SC_GHOST_BIT) return fail(ctx, "sc_set_state_uids: uids must be < 2^31");
        if (uid[i] > top) top = uid[i];
    }
    CKR(sc_set_state(ctx, pos, vel, n));
    if (n) CK(cudaMemcpyAsync(ctx->uid_cur, uid, sizeof(uint32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    CK(stream_sync(ctx));
    ctx->next_uid = top + 1;
    return 0;
}

extern "C" int sc_append_particles(sc_ctx *ctx, const double *pos, const double *vel, int64_t n) {
    CKR(enter(ctx, "sc_append_particles"));
    CKR(drop_keys(ctx));
    if (ctx->in_step) return fail(ctx, "sc_append_particles: inside a split step");
    if (n < 0) return fail(ctx, "sc_append_particles: n < 0");
    CKR(sync_count(ctx));
    if (ctx->n_host + n > ctx->cap) return fail(ctx, "sc_append_particles: capacity exceeded");
    ctx->srt_valid = false; ctx->lists_valid = false;  // (appended rows sit behind the sorted ones: rows_valid stays)
    return upload_particles(ctx, pos, vel, ctx->n_host, n);
}

extern "C" uint64_t sc_source_stream(uint64_t seed, uint64_t tick, uint32_t source_index, uint64_t j, double *u) {
    const uint64_t key = source_key(tick_key(seed, tick), source_index);
    if (u) *u = source_uniform(key, j);
    return key;
}

extern "C" int sc_emit_particles(sc_ctx *ctx, const sc_source *sources, int nsources, int64_t max_particles) {
    CKR(enter(ctx, "sc_emit_particles"));
    if (nsources > 0 && !sources) return fail(ctx, "sc_emit_particles: NULL argument");
    if (ctx->in_step) return fail(ctx, "sc_emit_particles: inside a split step");
    if (nsources < 0 || nsources > SC_MAX_SOURCES) return fail(ctx, "sc_emit_particles: more than SC_MAX_SOURCES sources");
    if (ctx->dist_on) return fail(ctx, "sc_emit_particles: strips support closed scenes only");
    EmitParams E{};
    E.nsrc = 0;
    E.max_particles = (uint32_t)std::min<int64_t>(std::max<int64_t>(max_particles, 0), ctx->cap);
    uint64_t total = 0;
    const uint64_t tkey = tick_key(ctx->seed, ctx->tick);
    for (int q = 0; q < nsources; ++q) {
        if (sources[q].count <= 0) continue;
        EmitSource &S = E.src[E.nsrc++];
        S.px = sources[q].position_x; S.py = sources[q].position_y; S.radius = sources[q].radius;
        S.vx = sources[q].velocity_x; S.vy = sources[q].velocity_y; S.vnoise = sources[q].velocity_noise;
        S.key = source_key(tkey, sources[q].index);
        S.n = (uint32_t)sources[q].count;
        S.uid_base = ctx->next_uid + (uint32_t)total;   // identities advance by the DRAWN count; a clamp leaves a gap
        total += S.n;
    }
    if (!E.nsrc) return 0;
    CKR(drop_keys(ctx));  // the new particles have no keys
    if ((uint64_t)ctx->next_uid + total >= (uint64_t)SC_GHOST_BIT)
        return fail(ctx, "particle identities exhausted (2^31 particles created in this context)");
    refresh_count(ctx);
    {
        ProfScope ps(ctx, SLOT_IO);
        if (ctx->precision == SC_PRECISION_F64)
            CK(launch_pdl(k_emit<double>, dim3(1), dim3(SC_BLOCK), ctx->stream, ctx->cnt, E, ctx->pos_cur, (double2 *)ctx->vel_cur,
                          ctx->uid_cur, (uint32_t)ctx->cap));
        else
            CK(launch_pdl(k_emit<float>, dim3(1), dim3(SC_BLOCK), ctx->stream, ctx->cnt, E, ctx->pos_cur, (float2 *)ctx->vel_cur,
                          ctx->uid_cur, (uint32_t)ctx->cap));
    }
    ctx->next_uid += (uint32_t)total;
    ctx->n_host = std::min<int64_t>(ctx->n_host + (int64_t)total, ctx->cap);  // an upper bound: the clamp happened on the device
    ctx->n_exact = false;
    ctx->srt_valid = false; ctx->lists_valid = false; ctx->rank_valid = false;
    return 0;
}

extern "C" int sc_host_alloc(size_t bytes, void **out) {
    if (!out) return fail(nullptr, "sc_host_alloc: out is NULL");
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(nullptr, std::string("sc_host_alloc: ") + cudaGetErrorString(e));
    return 0;
}
extern "C" int sc_host_free(void *p) {
    if (!p) return 0;
    cudaError_t e = cudaFreeHost(p);
    if (e != cudaSuccess) return fail(nullptr, std::string("sc_host_free: ") + cudaGetErrorString(e));
    return 0;
}

extern "C" int sc_particle_count(sc_ctx *ctx, int64_t *n) {
    CKR(enter(ctx, "sc_particle_count"));
    if (!n) return fail(ctx, "sc_particle_count: NULL argument");
    CKR(sync_count(ctx));
    *n = ctx->n_host;
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// Exclusive scan of in[0..n) to out[0..n), total to out[n] (in == out: in place).  `pre_cleared`: the descriptors were
// zeroed by k_begin_tick / the last force kernel.
static int exclusive_scan(sc_ctx *ctx, const uint32_t *in, uint32_t *out, uint32_t n, int slot, bool pre_cleared = false) {
    const unsigned nb = (n + SC_SCAN_TILE - 1) / SC_SCAN_TILE;
    if (nb == 0) { CK(cudaMemsetAsync(out, 0, sizeof(uint32_t), ctx->stream)); return 0; }
    // the cell scan's descriptors (bsum) are kept zeroed from tick to tick by the force kernel; every other scan uses
    // its own set and zeroes it here
    unsigned long long *&desc = pre_cleared ? ctx->bsum : ctx->bsum2;
    size_t &cap = pre_cleared ? ctx->bsum_cap : ctx->bsum2_cap;
    if ((size_t)nb + 2 > cap) {
        CK(stream_sync(ctx));
        if (desc) CK(cudaFree(desc));
        CKR(dev_alloc(ctx, &desc, (size_t)nb + 2));
        cap = (size_t)nb + 2;
        pre_cleared = false;
    }
    if (!pre_cleared) CK(cudaMemsetAsync(desc, 0, sizeof(unsigned long long) * ((size_t)nb + 1), ctx->stream));
    ProfScope ps(ctx, slot);
    CK(launch_pdl(k_scan_lookback, dim3(nb), dim3(SC_SCAN_THREADS), ctx->stream, in, out, n, desc + 1, (uint32_t *)desc));
    return 0;
}

// uid -> rank among live particles, for the uid array `uid` holding `cnt->n`-many... the live count is read from
// n_ptr on the device.
static int build_rank_map(sc_ctx *ctx, const uint32_t *uid, const uint32_t *n_ptr) {
    const size_t need = (size_t)ctx->next_uid + 2;
    if (need > ctx->uid_cap) {
        CK(stream_sync(ctx));
        if (ctx->rank_of_uid) CK(cudaFree(ctx->rank_of_uid));
        size_t cap = need * 2 > (size_t)ctx->cap + 2 ? need * 2 : (size_t)ctx->cap + 2;
        CKR(dev_alloc(ctx, &ctx->rank_of_uid, cap));
        ctx->uid_cap = cap;
    }
    CK(cudaMemsetAsync(ctx->rank_of_uid, 0, sizeof(uint32_t) * need, ctx->stream));
    if (ctx->n_host > 0) {
        ProfScope ps(ctx, SLOT_RANKMAP);
        k_mark_alive<<<blocks_for(ctx->n_host), SC_BLOCK, 0, ctx->stream>>>(n_ptr, uid, ctx->rank_of_uid);
    }
    CKR(exclusive_scan(ctx, ctx->rank_of_uid, ctx->rank_of_uid, ctx->next_uid, SLOT_RANKMAP));
    return 0;
}

static int require_ready(sc_ctx *ctx, const char *who, bool consumes_unpack = false) {
    CKR(enter(ctx, who, consumes_unpack));
    if (!ctx->params_set) return fail(ctx, std::string(who) + ": sc_set_params has not been called");
    return 0;
}

// where the key pass of a tick of parity `q` writes (key_particle, sc_common.cuh)
static KeyOut key_out(sc_ctx *ctx, int q) {
    return KeyOut{ctx->cell_key, ctx->cell_count, ctx->wbits_cur[q], ctx->wall_slot_cur, &ctx->cnt->n_wall[q],
                  ctx->pos_cur, ctx->wall_pre_buf[q]};
}

// remove -> walls -> keys -> sort -> gather
template <bool kStep> static int enqueue_search(sc_ctx *ctx) {
    const int64_t n = ctx->n_host;
    const Grid &g = ctx->grid;
    // this tick's wall set: the one the previous tick's density kernel cleared (and its force kernel may have filled)
    ctx->par ^= 1;
    ctx->wall_bits_cur = ctx->wbits_cur[ctx->par];
    ctx->wall_bits_srt = ctx->wbits_srt[ctx->par];
    ctx->wall_pre = ctx->wall_pre_buf[ctx->par];
    const bool keyed = kStep && ctx->next_keyed;  // the previous tick's force kernel did this tick's pre-pass
    if (!ctx->next_clean && !keyed) {  // cold start: first tick of the context / first after the grid was rebuilt
        CKR(launch_clear(ctx, ctx->par, ctx->carry_count ? ctx->cell_start + g.ncells : nullptr, KeyRestore{}));
        ctx->carry_count = false;
    }
    ctx->next_clean = false;
    ctx->next_keyed = false;
    // strips: a recorded (deferred) unpack is carried out by the pre-pass itself (PrepassUnpack, sc_common.cuh)
    PrepassUnpack U{};
    if (ctx->pend.on) {
        U.on = 1; U.vel_is_f64 = ctx->precision == SC_PRECISION_F64;
        U.lo = UnpackSide{ctx->dist.has_lo ? (const WireHeader *)ctx->pend.recv_lo : nullptr, (const uint32_t *)ctx->pend.flag_lo};
        U.hi = UnpackSide{ctx->dist.has_hi ? (const WireHeader *)ctx->pend.recv_hi : nullptr, (const uint32_t *)ctx->pend.flag_hi};
        U.value = ctx->pend.value; U.wire_cap = ctx->dist.cap;
        U.vel = ctx->vel_cur; U.uid = ctx->uid_cur;
        U.send_lo = ctx->send_lo ? ctx->send_lo : ctx->wire_dummy;
        U.send_hi = ctx->send_hi ? ctx->send_hi : ctx->wire_dummy + 1;
        if (!U.lo.hdr && !U.hi.hdr) U.on = 0;
        ctx->pend.on = false;
    }
    if (n > 0 && !keyed) {
        ProfScope ps(ctx, SLOT_PREPASS);
        auto go = [&](auto kernel) {
            return launch_pdl(kernel, dim3(blocks_for((n + SC_PREPASS_ILP - 1) / SC_PREPASS_ILP)), dim3(SC_BLOCK),
                              ctx->stream, ctx->cnt, g, ctx->dp, ctx->walls, key_out(ctx, ctx->par), (uint32_t)ctx->cap, U);
        };
        CK(U.on ? go(k_prepass<kStep, true>) : go(k_prepass<kStep, false>));
    }
    CKR(exclusive_scan(ctx, ctx->cell_count, ctx->cell_start, g.ncells, SLOT_SCAN, true));
    if (n > 0) {
        {
            ProfScope ps(ctx, SLOT_PLACE);
            CK(launch_pdl(k_place, dim3(blocks_for((n + SC_PLACE_ILP - 1) / SC_PLACE_ILP)), dim3(SC_BLOCK), ctx->stream,
                          (const Counters *)ctx->cnt, (const uint32_t *)ctx->cell_key, ctx->cell_count,
                          (const uint32_t *)ctx->cell_start, ctx->tmpidx, (uint32_t)ctx->cap));
        }
        ProfScope ps(ctx, SLOT_RANK_GATHER);
        if (ctx->precision == SC_PRECISION_F64)
            CK(launch_pdl(k_rank_gather<double>, dim3(blocks_for(n)), dim3(SC_BLOCK), ctx->stream,
                ctx->cnt, g, ctx->cell_start, ctx->tmpidx, ctx->cell_key, ctx->pos_cur, (const double2 *)ctx->vel_cur,
                ctx->uid_cur, ctx->wall_bits_cur, ctx->wall_slot_cur, ctx->pos_srt, ctx->rel_srt, (double2 *)ctx->vel_srt,
                ctx->uid_srt, ctx->cell_key_srt, ctx->wall_bits_srt, ctx->wall_slot_srt, (float4 *)nullptr, (BlockDesc *)nullptr));
        else
            CK(launch_pdl(k_rank_gather<float>, dim3(blocks_for(n)), dim3(SC_BLOCK), ctx->stream,
                ctx->cnt, g, ctx->cell_start, ctx->tmpidx, ctx->cell_key, ctx->pos_cur, (const float2 *)ctx->vel_cur,
                ctx->uid_cur, ctx->wall_bits_cur, ctx->wall_slot_cur, ctx->pos_srt, ctx->rel_srt, (float2 *)ctx->vel_srt,
                ctx->uid_srt, ctx->cell_key_srt, ctx->wall_bits_srt, ctx->wall_slot_srt, ctx->rec_srt, ctx->blk_desc));
    }
    CK(cudaGetLastError());
    ctx->srt_valid = true;
    ctx->lists_valid = false;
    ctx->rank_valid = false;
    return 0;
}

// After enqueue_forces the uids of the sorted set live in uid_cur (pointer swap); inside a split step they are
// still in uid_srt.
static inline const uint32_t *sorted_uids(const sc_ctx *c) { return c->in_step ? c->uid_srt : c->uid_cur; }

// rank map + neighbor counts (+ lists) for the sorted set
static int enqueue_count(sc_ctx *ctx, const uint32_t *uid, bool want_lists) {
    const int64_t n = ctx->n_host;
    const uint32_t *n_ptr = ctx->cell_start + ctx->grid.ncells;
    if (!ctx->rank_valid) { CKR(build_rank_map(ctx, uid, n_ptr)); ctx->rank_valid = true; }
    if (want_lists && !ctx->list_sorted) {
        CKR(dev_alloc(ctx, &ctx->list_sorted, (size_t)ctx->cap * SC_MAX_NEIGHBORS));
    }
    CK(cudaMemsetAsync(&ctx->cnt->n_pairs, 0, sizeof(uint32_t), ctx->stream));
    if (n > 0) {
        ProfScope ps(ctx, SLOT_COUNT);
        k_count_neighbors<<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(
            ctx->cnt, ctx->grid, ctx->cell_start, ctx->pos_srt, ctx->rel_srt, ctx->cell_key_srt, uid, ctx->rank_of_uid,
            ctx->count_by_rank, want_lists ? ctx->list_sorted : nullptr);
    }
    CK(cudaGetLastError());
    ctx->lists_valid = want_lists;
    return 0;
}

// what this tick's density kernel clears for the next tick (NextWallClear, sc_common.cuh)
static NextWallClear next_wall_clear(sc_ctx *ctx) {
    const int o = ctx->par ^ 1;
    return NextWallClear{ctx->wbits_cur[o], ctx->wbits_srt[o], (uint32_t)(ctx->cap / 32 + 1), &ctx->cnt->n_wall[o]};
}

static int launch_density(sc_ctx *ctx, const DevParams &dp, const uint32_t *noise_off, int64_t n) {
    auto go = [&](auto kernel) {
        return launch_pdl(kernel, dim3(blocks_for(n)), dim3(SC_BLOCK), ctx->stream, ctx->cnt, ctx->grid, dp, ctx->cell_start,
                          ctx->pos_srt, ctx->rel_srt, ctx->cell_key_srt, ctx->uid_cur, ctx->noise_dev, noise_off,
                          ctx->rank_of_uid, ctx->pair_j, (double2 *)ctx->pair_n, ctx->pair_off, ctx->pair_cnt,
                          (PS<double> *)ctx->ps, next_wall_clear(ctx));
    };
    if (dp.noise_mode == SC_NOISE_HOST) CK(go(k_density<SC_NOISE_HOST>));
    else if (dp.noise_mode == SC_NOISE_COUNTER) CK(go(k_density<SC_NOISE_COUNTER>));
    else CK(go(k_density<SC_NOISE_NONE>));
    return 0;
}

// K4 stages the block's neighborhood in shared memory (sc_tile.cuh)
static int launch_density_tile(sc_ctx *ctx, const DevParams &dp, const uint32_t *noise_off, int64_t n) {
    auto go = [&](auto kernel) {
        return launch_pdl(kernel, dim3((unsigned)((n + SC_TILE - 1) / SC_TILE)), dim3(SC_TILE), ctx->stream, ctx->cnt,
                          ctx->grid, dp, ctx->cell_start, ctx->blk_desc, ctx->pos_srt, ctx->rec_srt, ctx->cell_key_srt,
                          (uint2 *)ctx->pair_n, ctx->pair_cnt, (PS<float> *)ctx->ps, next_wall_clear(ctx),
                          HostNoise{ctx->noise_dev, noise_off, ctx->rank_of_uid});
    };
    if (dp.noise_mode == SC_NOISE_HOST) CK(go(k_density_tile<SC_NOISE_HOST>));
    else if (dp.noise_mode == SC_NOISE_COUNTER) CK(go(k_density_tile<SC_NOISE_COUNTER>));
    else CK(go(k_density_tile<SC_NOISE_NONE>));
    return 0;
}

// what this tick's force kernel does for the next tick (TickDuty, sc_common.cuh), and the next tick's key pass when
// `keys` (NextKeys, sc_pair.cuh)
static TickDuty tick_duty(sc_ctx *ctx) {
    TickDuty d;
    d.scan_desc = ctx->bsum; d.scan_words = (ctx->grid.ncells + SC_SCAN_TILE - 1) / SC_SCAN_TILE + 1;
    d.cnt = ctx->cnt;
    return d;
}
static NextKeys next_keys(sc_ctx *ctx, bool keys) {
    NextKeys k{};
    k.g = ctx->grid;
    if (keys) k.out = key_out(ctx, ctx->par ^ 1);
    return k;
}

static int launch_force(sc_ctx *ctx, const DevParams &dp, const uint32_t *n_ptr, int64_t n, bool keys) {
    const unsigned nb = (unsigned)((n + SC_K5_THREADS - 1) / SC_K5_THREADS);
    auto go = [&](auto kernel) {
        return launch_pdl(kernel, dim3(nb), dim3(SC_K5_THREADS), ctx->stream, n_ptr, dp, ctx->walls, ctx->pos_srt,
                          (const double2 *)ctx->vel_srt, ctx->pair_j, (const double2 *)ctx->pair_n, ctx->pair_off,
                          ctx->pair_cnt, (const PS<double> *)ctx->ps, ctx->wall_bits_srt, ctx->wall_slot_srt,
                          ctx->wall_pre, ctx->pos_cur, (double2 *)ctx->vel_cur, ctx->monitor, tick_duty(ctx),
                          next_keys(ctx, keys));
    };
    CK(ctx->monitor_on ? go(k_force<true>) : go(k_force<false>));
    return 0;
}

// K5 on the same blocks and windows as K4 (sc_tile.cuh)
static int launch_force_tile(sc_ctx *ctx, const DevParams &dp, const uint32_t *n_ptr, int64_t n, bool keys) {
    auto go = [&](auto kernel) {
        return launch_pdl(kernel, dim3((unsigned)((n + SC_TILE - 1) / SC_TILE)), dim3(SC_TILE), ctx->stream, n_ptr, dp,
                          ctx->walls, ctx->blk_desc, ctx->pos_srt, (const float2 *)ctx->vel_srt, (const uint2 *)ctx->pair_n,
                          ctx->pair_cnt, (const PS<float> *)ctx->ps, ctx->wall_bits_srt, ctx->wall_slot_srt,
                          ctx->wall_pre, ctx->pos_cur, (float2 *)ctx->vel_cur, ctx->monitor, tick_duty(ctx),
                          next_keys(ctx, keys));
    };
    CK(ctx->monitor_on ? go(k_force_tile<true>) : go(k_force_tile<false>));
    return 0;
}

// The parameters of the step of tick `tick`: its noise key, and the effective noise mode (a zero noise level is none).
static DevParams step_params(const sc_ctx *ctx, uint64_t tick) {
    DevParams dp = ctx->dp;
    dp.noise_mode = (ctx->noise_mode != SC_NOISE_NONE && ctx->hp.collider_noise_level == 0.0) ? SC_NOISE_NONE
                                                                                             : ctx->noise_mode;
    dp.tick_key = tick_key(ctx->seed, tick);
    return dp;
}

// The pair kernels of the last search, chosen by the precision alone: k_density / k_force (sc_pair.cuh) in fp64, the
// tiled kernels (sc_tile.cuh) in mixed precision, in every noise mode.  `k4`, `k5`: which of the two to enqueue.
// `noise_off`: the CSR offsets of SC_NOISE_HOST.  The sorted set's uids must be in uid_cur.
static int launch_pair_kernels(sc_ctx *ctx, const DevParams &dp, const uint32_t *noise_off, bool k4, bool k5, bool keys) {
    const int64_t n = ctx->n_host;
    const bool f64 = ctx->precision == SC_PRECISION_F64;
    if (k4) {
        ProfScope ps(ctx, SLOT_DENSITY);
        CKR(f64 ? launch_density(ctx, dp, noise_off, n) : launch_density_tile(ctx, dp, noise_off, n));
    }
    if (k5) {
        if (ctx->monitor_on) CK(cudaMemsetAsync(ctx->monitor, 0, sizeof(double) * 8, ctx->stream));
        ProfScope ps(ctx, SLOT_FORCE);
        const uint32_t *n_ptr = ctx->cell_start + ctx->grid.ncells;
        CKR(f64 ? launch_force(ctx, dp, n_ptr, n, keys) : launch_force_tile(ctx, dp, n_ptr, n, keys));
    }
    return 0;
}

static int enqueue_forces(sc_ctx *ctx, const uint32_t *noise_off) {
    const int64_t n = ctx->n_host;
    // the new state (pos_cur, vel_cur) is in this tick's sorted order, whose uids are uid_srt
    uint32_t *t = ctx->uid_cur; ctx->uid_cur = ctx->uid_srt; ctx->uid_srt = t;
    // the force kernel runs the next tick's key pass (NextKeys) unless a call since the last step changed what the keys
    // depend on (drop_keys) or this is a strip, whose exchange changes the particle set between the ticks
    const bool keys = n > 0 && !ctx->keys_dropped && !ctx->dist_on;
    if (n > 0) CKR(launch_pair_kernels(ctx, step_params(ctx, ctx->tick), noise_off, true, true, keys));
    // the force kernel carried the count; the density kernel cleared the next tick's wall set, k_place the counts
    if (n > 0) { ctx->next_clean = !keys; ctx->next_keyed = keys; ctx->carry_count = false; }
    else ctx->carry_count = true;  // nothing ran: cnt->n is refreshed by the next cold start or by sync_count
    ctx->keys_dropped = false;
    CK(cudaGetLastError());
    ctx->rows_valid = n > 0;
    ctx->tick += 1;  // crate.py:127
    ctx->n_exact = false;
    return 0;
}

extern "C" int sc_step(sc_ctx *ctx) {
    CKR(require_ready(ctx, "sc_step", true));
    if (ctx->in_step) return fail(ctx, "sc_step: a split step is open");
    if (ctx->noise_mode == SC_NOISE_HOST && ctx->hp.collider_noise_level != 0.0)
        return fail(ctx, "sc_step: SC_NOISE_HOST needs sc_step_begin / sc_step_finish");
    CKR(enqueue_search<true>(ctx));
    return enqueue_forces(ctx, nullptr);
}

extern "C" int sc_step_n(sc_ctx *ctx, int nsteps) {
    for (int i = 0; i < nsteps; ++i) CKR(sc_step(ctx));
    return 0;
}

extern "C" int sc_step_begin(sc_ctx *ctx, int64_t *n_particles, int64_t *n_pairs) {
    CKR(require_ready(ctx, "sc_step_begin", true));
    if (ctx->in_step) return fail(ctx, "sc_step_begin: a split step is already open");
    CKR(enqueue_search<true>(ctx));
    ctx->in_step = true;
    CKR(enqueue_count(ctx, ctx->uid_srt, false));
    Counters h;
    uint32_t total = 0;
    CK(cudaMemcpyAsync(&h, ctx->cnt, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&total, ctx->cell_start + ctx->grid.ncells, sizeof(uint32_t), cudaMemcpyDeviceToHost,
                       ctx->stream));
    CK(stream_sync(ctx));
    if (n_particles) *n_particles = total;
    if (n_pairs) *n_pairs = h.n_pairs;
    return 0;
}

extern "C" int sc_step_finish(sc_ctx *ctx, const double *noise) {
    CKR(require_ready(ctx, "sc_step_finish"));
    if (!ctx->in_step) return fail(ctx, "sc_step_finish: no split step is open");
    const uint32_t *noise_off = nullptr;
    const bool host_noise = ctx->noise_mode == SC_NOISE_HOST && ctx->hp.collider_noise_level != 0.0;
    if (host_noise) {
        if (!noise) return fail(ctx, "sc_step_finish: SC_NOISE_HOST needs the noise array");
        Counters h;
        CK(cudaMemcpyAsync(&h, ctx->cnt, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
        CK(stream_sync(ctx));
        const size_t need = (size_t)h.n_pairs * 2;
        if (need > ctx->noise_cap) {
            if (ctx->noise_dev) CK(cudaFree(ctx->noise_dev));
            CKR(dev_alloc(ctx, &ctx->noise_dev, need * 2 + 64));
            ctx->noise_cap = need * 2 + 64;
        }
        if (need) CK(cudaMemcpyAsync(ctx->noise_dev, noise, sizeof(double) * need, cudaMemcpyHostToDevice, ctx->stream));
        // CSR offsets in original index order (crate.py:165: `for particle_index in range(self.particle_count)`)
        CKR(exclusive_scan(ctx, ctx->count_by_rank, ctx->count_by_rank, (uint32_t)ctx->n_host, SLOT_COUNT));
        noise_off = ctx->count_by_rank;
        ctx->lists_valid = false;
    }
    ctx->in_step = false;
    CKR(enqueue_forces(ctx, noise_off));
    if (host_noise) CK(stream_sync(ctx));  // `noise` is borrowed for the call only
    return 0;
}

extern "C" int sc_synchronize(sc_ctx *ctx) {
    if (!ctx) return fail(ctx, "sc_synchronize: NULL ctx");
    CK(cudaSetDevice(ctx->device));
    CK(stream_sync(ctx));
    CK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// readback (original index order)
// The uid -> row map is sized from THIS context's uids.  A strip with neighbors also holds ghosts (bit 31 set) and
// migrants with other ranks' uids, which would index far outside it: those contexts read back through
// sc_dist_get_owned instead.
static int no_neighbors(sc_ctx *ctx, const char *who) {
    if (ctx->dist_on && (ctx->dist.has_lo || ctx->dist.has_hi))
        return fail(ctx, std::string(who) + ": not available on a strip with neighbors (use sc_dist_get_owned)");
    return 0;
}
static int ensure_rank_for_current(sc_ctx *ctx) {
    // the current state's uid array is uid_cur and its live count is cnt->n
    if (!ctx->rank_valid) {
        CKR(build_rank_map(ctx, sorted_uids(ctx), ctx->in_step ? ctx->cell_start + ctx->grid.ncells : &ctx->cnt->n));
        ctx->rank_valid = true;
    }
    return 0;
}

extern "C" int sc_get_state(sc_ctx *ctx, double *pos, double *vel, double *pressure, int64_t cap, int64_t *n_out) {
    CKR(enter(ctx, "sc_get_state"));
    if (ctx->in_step) return fail(ctx, "sc_get_state: inside a split step");
    CKR(no_neighbors(ctx, "sc_get_state"));
    CKR(sync_count(ctx));
    const int64_t n = ctx->n_host;
    if (n_out) *n_out = n;
    if (n > cap) return fail(ctx, "sc_get_state: buffer too small");
    if (n == 0) return 0;
    CKR(ensure_rank_for_current(ctx));
    const uint32_t *n_ptr = &ctx->cnt->n;
    const unsigned nb = blocks_for(n);
    if (pos) {
        const int q = ctx->par ^ 1;  // the wall set the next tick's key pass filled, if it ran (next_keyed)
        { ProfScope ps(ctx, SLOT_IO);
          k_scatter_pos<<<nb, SC_BLOCK, 0, ctx->stream>>>(n_ptr, ctx->uid_cur, ctx->rank_of_uid, ctx->pos_cur,
                                                          ctx->next_keyed ? ctx->wbits_cur[q] : nullptr, ctx->wall_slot_cur,
                                                          ctx->wall_pre_buf[q], ctx->stage2); }
        CK(cudaMemcpyAsync(pos, ctx->stage2, sizeof(double2) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (vel) {
        { ProfScope ps(ctx, SLOT_IO);
          if (ctx->precision == SC_PRECISION_F64)
              k_scatter_vec2<double2><<<nb, SC_BLOCK, 0, ctx->stream>>>(n_ptr, ctx->uid_cur, ctx->rank_of_uid, (const double2 *)ctx->vel_cur, ctx->stage2);
          else
              k_scatter_vec2<float2><<<nb, SC_BLOCK, 0, ctx->stream>>>(n_ptr, ctx->uid_cur, ctx->rank_of_uid, (const float2 *)ctx->vel_cur, ctx->stage2); }
        CK(cudaMemcpyAsync(vel, ctx->stage2, sizeof(double2) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (pressure) {
        if (!ctx->srt_valid) {
            CK(cudaMemsetAsync(ctx->stage1, 0, sizeof(double) * (size_t)n, ctx->stream));  // crate.py:26 before any tick
        } else {
            ProfScope ps(ctx, SLOT_IO);
            if (ctx->precision == SC_PRECISION_F64)
                k_scatter_ps<double><<<nb, SC_BLOCK, 0, ctx->stream>>>(n_ptr, ctx->uid_cur, ctx->rank_of_uid, (const PS<double> *)ctx->ps, ctx->stage1, nullptr);
            else
                k_scatter_ps<float><<<nb, SC_BLOCK, 0, ctx->stream>>>(n_ptr, ctx->uid_cur, ctx->rank_of_uid, (const PS<float> *)ctx->ps, ctx->stage1, nullptr);
        }
        CK(cudaMemcpyAsync(pressure, ctx->stage1, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(stream_sync(ctx));
    CK(cudaGetLastError());
    return 0;
}

extern "C" int sc_get_uids(sc_ctx *ctx, uint32_t *uid, int64_t cap, int64_t *n_out) {
    CKR(enter(ctx, "sc_get_uids"));
    if (ctx->in_step) return fail(ctx, "sc_get_uids: inside a split step");
    CKR(no_neighbors(ctx, "sc_get_uids"));
    CKR(sync_count(ctx));
    const int64_t n = ctx->n_host;
    if (n_out) *n_out = n;
    if (n > cap) return fail(ctx, "sc_get_uids: buffer too small");
    if (n == 0) return 0;
    CKR(ensure_rank_for_current(ctx));
    { ProfScope ps(ctx, SLOT_IO);
      k_scatter_uid<<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(&ctx->cnt->n, ctx->uid_cur, ctx->rank_of_uid, (uint32_t *)ctx->stage1); }
    CK(cudaMemcpyAsync(uid, ctx->stage1, sizeof(uint32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    return 0;
}

// ---- taps --------------------------------------------------------------------------------------------------
static int tap_prologue(sc_ctx *ctx, const char *who, int64_t cap, int64_t *n_out) {
    CKR(enter(ctx, who));
    if (!ctx->srt_valid) return fail(ctx, std::string(who) + ": no search state (call sc_step or sc_step_begin first)");
    CKR(no_neighbors(ctx, who));
    uint32_t total = 0;
    CK(cudaMemcpyAsync(&total, ctx->cell_start + ctx->grid.ncells, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    if ((int64_t)total > cap) return fail(ctx, std::string(who) + ": buffer too small");
    *n_out = total;
    if (!ctx->rank_valid) {
        CKR(build_rank_map(ctx, sorted_uids(ctx), ctx->cell_start + ctx->grid.ncells));
        ctx->rank_valid = true;
    }
    return 0;
}

extern "C" int sc_get_search(sc_ctx *ctx, double *pos_search, int64_t *rows_sorted, int64_t *order, int64_t cap) {
    int64_t n = 0;
    CKR(tap_prologue(ctx, "sc_get_search", cap, &n));
    if (n == 0) return 0;
    const uint32_t *n_ptr = ctx->cell_start + ctx->grid.ncells;
    const uint32_t *uid = sorted_uids(ctx);
    if (pos_search) {
        { ProfScope ps(ctx, SLOT_IO);
          k_scatter_vec2<double2><<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(n_ptr, uid, ctx->rank_of_uid, ctx->pos_srt, ctx->stage2); }
        CK(cudaMemcpyAsync(pos_search, ctx->stage2, sizeof(double2) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
        CK(stream_sync(ctx));
    }
    if (rows_sorted || order) {
        long long *rows_d = (long long *)ctx->stage2, *order_d = rows_d + n;  // stage2 holds 2n 8-byte slots
        { ProfScope ps(ctx, SLOT_IO);
          k_tap_search<<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(n_ptr, ctx->grid, ctx->pos_srt, uid, ctx->rank_of_uid, rows_d, order_d); }
        if (rows_sorted) CK(cudaMemcpyAsync(rows_sorted, rows_d, sizeof(int64_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
        if (order) CK(cudaMemcpyAsync(order, order_d, sizeof(int64_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
        CK(stream_sync(ctx));
    }
    CK(cudaGetLastError());
    return 0;
}

extern "C" int sc_get_neighbors(sc_ctx *ctx, int32_t *counts, int32_t *idx, int64_t cap) {
    int64_t n = 0;
    CKR(tap_prologue(ctx, "sc_get_neighbors", cap, &n));
    if (n == 0) return 0;
    // (re)run the count kernel on the sorted set with list output; count_by_rank may hold CSR offsets after a
    // host-noise finish, so it is always rebuilt here
    CKR(enqueue_count(ctx, sorted_uids(ctx), true));
    const uint32_t *n_ptr = ctx->cell_start + ctx->grid.ncells;
    if (counts) CK(cudaMemcpyAsync(counts, ctx->count_by_rank, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (idx) {
        int *idx_d = nullptr;
        CK(cudaMalloc((void **)&idx_d, sizeof(int) * (size_t)n * SC_MAX_NEIGHBORS));
        { ProfScope ps(ctx, SLOT_IO);
          k_tap_lists<<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(n_ptr, sorted_uids(ctx), ctx->rank_of_uid, ctx->count_by_rank, ctx->list_sorted, idx_d); }
        CK(cudaMemcpyAsync(idx, idx_d, sizeof(int) * (size_t)n * SC_MAX_NEIGHBORS, cudaMemcpyDeviceToHost, ctx->stream));
        CK(stream_sync(ctx));
        CK(cudaFree(idx_d));
    }
    CK(stream_sync(ctx));
    CK(cudaGetLastError());
    return 0;
}

extern "C" int sc_get_tension(sc_ctx *ctx, double *tension, int64_t cap) {
    int64_t n = 0;
    CKR(tap_prologue(ctx, "sc_get_tension", cap, &n));
    if (n == 0 || !tension) return 0;
    if (ctx->in_step) return fail(ctx, "sc_get_tension: inside a split step");
    const uint32_t *n_ptr = ctx->cell_start + ctx->grid.ncells;
    { ProfScope ps(ctx, SLOT_IO);
      if (ctx->precision == SC_PRECISION_F64)
          k_scatter_ps<double><<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(n_ptr, sorted_uids(ctx), ctx->rank_of_uid, (const PS<double> *)ctx->ps, nullptr, ctx->stage2);
      else
          k_scatter_ps<float><<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(n_ptr, sorted_uids(ctx), ctx->rank_of_uid, (const PS<float> *)ctx->ps, nullptr, ctx->stage2); }
    CK(cudaMemcpyAsync(tension, ctx->stage2, sizeof(double2) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    CK(cudaGetLastError());
    return 0;
}

extern "C" int sc_get_wall_counts(sc_ctx *ctx, int32_t *counts, int64_t cap) {
    int64_t n = 0;
    CKR(tap_prologue(ctx, "sc_get_wall_counts", cap, &n));
    if (n == 0 || !counts) return 0;
    const uint32_t *n_ptr = ctx->cell_start + ctx->grid.ncells;
    { ProfScope ps(ctx, SLOT_IO);
      k_tap_wall_counts<<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(n_ptr, ctx->dp, ctx->walls, sorted_uids(ctx), ctx->rank_of_uid, ctx->wall_bits_srt, ctx->wall_slot_srt, ctx->wall_pre, (int *)ctx->stage1); }
    CK(cudaMemcpyAsync(counts, ctx->stage1, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    CK(cudaGetLastError());
    return 0;
}

// ---- standalone layer-2 ops ----------------------------------------------------------------------------------
extern "C" int sc_detect_particle_collisions(sc_ctx *parent, const double *particles, int64_t P, double diameter,
                                             int64_t *rows_sorted, int64_t *order, int32_t *counts, int32_t *idx) {
    CKR(enter(parent, "sc_detect_particle_collisions"));
    if (P < 0 || !(diameter > 0)) return fail(parent, "sc_detect_particle_collisions: bad arguments");
    if (P == 0) return 0;
    // a private context keeps the caller's simulation state untouched
    sc_ctx *t = nullptr;
    if (sc_create(parent->device, SC_PRECISION_F64, P, nullptr, &t)) return fail(parent, g_create_error);
    auto bail = [&](int rc) { if (rc) parent->err = t->err; sc_destroy(t); return rc; };
    int rc = 0;
    do {
        t->hp = sc_params{}; t->hp.particle_radius = diameter / 2; t->params_set = true;
        refresh_dev_params(t);
        t->dp.d = diameter;  // r * 2 would round differently for odd diameters; the search only uses d
        std::vector<double> zeros((size_t)P * 2, 0.0);
        // grid bounds from the data
        int hb[4] = {INT32_MAX, INT32_MIN, INT32_MAX, INT32_MIN};
        int *db = nullptr;
        if (cudaMalloc((void **)&db, sizeof(hb)) != cudaSuccess) { rc = fail(t, "cudaMalloc bounds"); break; }
        cudaMemcpyAsync(db, hb, sizeof(hb), cudaMemcpyHostToDevice, t->stream);
        // upload without a grid yet
        t->grid.d = diameter; t->grid.inv_d = 1.0 / diameter;
        if ((rc = upload_particles(t, particles, zeros.data(), 0, P))) { cudaFree(db); break; }
        k_cell_bounds<<<blocks_for(P), SC_BLOCK, 0, t->stream>>>(t->pos_cur, (uint32_t)P, diameter, db);
        cudaMemcpyAsync(hb, db, sizeof(hb), cudaMemcpyDeviceToHost, t->stream);
        cudaStreamSynchronize(t->stream);
        cudaFree(db);
        if ((rc = setup_grid(t, diameter, hb[0], hb[1], hb[2], hb[3]))) break;
        if ((rc = enqueue_search<false>(t))) break;
        t->in_step = true;  // sorted uids are in uid_srt
        int64_t n = 0;
        if ((rc = tap_prologue(t, "sc_detect_particle_collisions", P, &n))) break;
        if ((rc = sc_get_search(t, nullptr, rows_sorted, order, P))) break;
        if ((rc = sc_get_neighbors(t, counts, idx, P))) break;
    } while (0);
    parent->launches += t->launches;
    return bail(rc);
}

extern "C" int sc_points_to_segments_distance(sc_ctx *ctx, const double *p, int64_t P, const double *segments, int S,
                                              double *nearest, double *dist) {
    CKR(enter(ctx, "sc_points_to_segments_distance"));
    if (P < 0 || S < 0) return fail(ctx, "sc_points_to_segments_distance: bad arguments");
    if (P == 0 || S == 0) return 0;
    if (P * (int64_t)S > ((int64_t)1 << 31) - 1) return fail(ctx, "sc_points_to_segments_distance: P*S too large");
    double2 *dp = nullptr; double *ds = nullptr, *dn = nullptr, *dd = nullptr;
    CK(cudaMalloc((void **)&dp, sizeof(double2) * (size_t)P));
    CK(cudaMalloc((void **)&ds, sizeof(double) * 4 * (size_t)S));
    CK(cudaMalloc((void **)&dn, sizeof(double) * 2 * (size_t)P * S));
    CK(cudaMalloc((void **)&dd, sizeof(double) * (size_t)P * S));
    CK(cudaMemcpyAsync(dp, p, sizeof(double2) * (size_t)P, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ds, segments, sizeof(double) * 4 * (size_t)S, cudaMemcpyHostToDevice, ctx->stream));
    { ProfScope ps(ctx, SLOT_IO);
      k_points_segments<<<blocks_for(P * S), SC_BLOCK, 0, ctx->stream>>>(dp, (uint32_t)P, ds, S, dn, dd); }
    if (nearest) CK(cudaMemcpyAsync(nearest, dn, sizeof(double) * 2 * (size_t)P * S, cudaMemcpyDeviceToHost, ctx->stream));
    if (dist) CK(cudaMemcpyAsync(dist, dd, sizeof(double) * (size_t)P * S, cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    CK(cudaGetLastError());
    cudaFree(dp); cudaFree(ds); cudaFree(dn); cudaFree(dd);
    return 0;
}

// directed pairs sum(K_i) of the last tick over the particles this context holds (ghosts included), = the number of
// pair records the density kernel handed to the force kernel.  Synchronises.
extern "C" int sc_last_pair_count(sc_ctx *ctx, int64_t *n_pairs) {
    CKR(enter(ctx, "sc_last_pair_count"));
    if (!n_pairs) return fail(ctx, "sc_last_pair_count: NULL argument");
    if (!ctx->srt_valid) { *n_pairs = 0; return 0; }
    CK(cudaMemsetAsync(&ctx->cnt->n_pairs, 0, sizeof(uint32_t), ctx->stream));
    if (ctx->n_host > 0) {
        ProfScope ps(ctx, SLOT_COUNT);
        k_sum_pair_counts<<<blocks_for(ctx->n_host), SC_BLOCK, 0, ctx->stream>>>(ctx->cell_start + ctx->grid.ncells,
                                                                                ctx->pair_cnt, &ctx->cnt->n_pairs);
    }
    Counters h;
    CK(cudaMemcpyAsync(&h, ctx->cnt, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    *n_pairs = (int64_t)h.n_pairs;
    return 0;
}

// ---- pair-record tap (declared in include/sandcrate.h under "diagnostics"): what the last tick's density kernel handed
// to its force kernel, per particle in original index order - K, the neighbors' row indices in list order, and the unit
// vectors as the force kernel decodes them.  It reads the pair buffers, so it must come before anything that rewrites
// them (the next step, sc_debug_rerun); inside a split step they still hold the tick before.
extern "C" int sc_debug_pair_records(sc_ctx *ctx, int32_t *counts, int32_t *nbr_row, double *nvec, int64_t cap) {
    int64_t n = 0;
    CKR(tap_prologue(ctx, "sc_debug_pair_records", cap, &n));
    if (ctx->in_step) return fail(ctx, "sc_debug_pair_records: inside a split step (the records are the last tick's)");
    if (n == 0) return 0;
    const size_t nr = (size_t)n * SC_MAX_NEIGHBORS;
    char *out_d = nullptr;  // [vectors nr x 16 | rows nr x 4 | counts n x 4]
    CK(cudaMalloc((void **)&out_d, nr * 16 + nr * 4 + (size_t)n * 4));
    double2 *vec_d = reinterpret_cast<double2 *>(out_d);
    int *row_d = reinterpret_cast<int *>(out_d + nr * 16), *cnt_d = row_d + nr;
    { ProfScope ps(ctx, SLOT_IO);
      k_tap_pair_records<<<(unsigned)((n + SC_TILE - 1) / SC_TILE), SC_TILE, 0, ctx->stream>>>(
          ctx->cell_start + ctx->grid.ncells, ctx->precision == SC_PRECISION_F64, ctx->blk_desc, ctx->pair_cnt,
          ctx->pair_off, ctx->pair_j, ctx->pair_n, sorted_uids(ctx), ctx->rank_of_uid, cnt_d, row_d, vec_d); }
    if (counts) CK(cudaMemcpyAsync(counts, cnt_d, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (nbr_row) CK(cudaMemcpyAsync(nbr_row, row_d, sizeof(int32_t) * nr, cudaMemcpyDeviceToHost, ctx->stream));
    if (nvec) CK(cudaMemcpyAsync(nvec, vec_d, sizeof(double2) * nr, cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    CK(cudaFree(out_d));
    CK(cudaGetLastError());
    return 0;
}

// the cell grid of the last search: origin row / column (the cell of (row, col) is (row - row_min) * ncols + col -
// col_min, clamped into [1, nrows - 2] x [1, ncols - 2]) and its size
extern "C" int sc_debug_grid(sc_ctx *ctx, int64_t *grid4) {
    CKR(enter(ctx, "sc_debug_grid"));
    if (!grid4) return fail(ctx, "sc_debug_grid: NULL argument");
    if (!ctx->params_set) return fail(ctx, "sc_debug_grid: sc_set_params has not been called");
    grid4[0] = ctx->grid.row_min; grid4[1] = ctx->grid.col_min; grid4[2] = ctx->grid.nrows; grid4[3] = ctx->grid.ncols;
    return 0;
}

// the conservative wall culls refresh_wall_boxes derived from the last sc_set_walls / radius (WallParams)
extern "C" int sc_debug_walls(sc_ctx *ctx, double *rects, double *seg_box, double *pad_box, int32_t *counts) {
    CKR(enter(ctx, "sc_debug_walls"));
    if (!ctx->walls_set) return fail(ctx, "sc_debug_walls: sc_set_walls has not been called");
    const WallParams &w = ctx->walls;
    if (rects)
        for (int q = 0; q < 4; ++q) {
            rects[q] = w.safe_contact[q]; rects[4 + q] = w.safe_ccd[q]; rects[8 + q] = (double)w.safe_ccd_f32[q];
        }
    if (seg_box && w.S) std::memcpy(seg_box, &w.seg_box[0][0], sizeof(double) * 4 * (size_t)w.S);
    if (pad_box && w.S) std::memcpy(pad_box, &w.pad_box[0][0], sizeof(double) * 8 * (size_t)w.S);
    if (counts) { counts[0] = w.S; counts[1] = ctx->grid_contacts; }
    return 0;
}

// ---- developer aids (declared in include/sandcrate.h under "diagnostics"): re-run one pair kernel of the last tick
// `reps` times and return the mean milliseconds.  K4 and K5 only read the sorted set, so re-running them is harmless.
// -1 before a step, inside a split step, and under SC_NOISE_HOST: the step's noise offsets live in count_by_rank, which
// the next count kernel (sc_get_neighbors, say) overwrites.
extern "C" double sc_debug_rerun(sc_ctx *ctx, int which, int reps) {
    if (!ctx || !ctx->srt_valid || ctx->in_step) return -1.0;
    const DevParams dp = step_params(ctx, ctx->tick - 1);
    if (dp.noise_mode == SC_NOISE_HOST) return -1.0;
    cudaSetDevice(ctx->device);
    if (drop_keys(ctx)) return -1.0;  // the force kernel re-run below computes no keys, and its own must not be counted twice
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float total = 0;
    for (int r = 0; r < reps; ++r) {
        if (which == 4) cudaMemsetAsync(&ctx->cnt->pair_cursor, 0, 4, ctx->stream);  // the fp64 K4 allocates from zero
        cudaEventRecord(e0, ctx->stream);
        launch_pair_kernels(ctx, dp, nullptr, which == 4, which != 4, false);
        cudaEventRecord(e1, ctx->stream);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        total += ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return total / reps;
}

// developer aid: how many blocks of the tiled density kernel took the pass-through path in the last tick
extern "C" int64_t sc_debug_untiled_blocks(sc_ctx *ctx) {
    if (!ctx) return -1;
    cudaSetDevice(ctx->device);
    Counters h;
    if (cudaMemcpyAsync(&h, ctx->cnt, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -1;
    return (int64_t)h.n_untiled;
}

// ---- ForceMonitor (utils/force_monitor.py) ------------------------------------------------------------------------
extern "C" int sc_set_monitor(sc_ctx *ctx, int on) {
    CKR(enter(ctx, "sc_set_monitor"));
    if (on && !ctx->monitor) {
        CKR(dev_alloc(ctx, &ctx->monitor, 8));
        CK(cudaMemsetAsync(ctx->monitor, 0, sizeof(double) * 8, ctx->stream));
    }
    ctx->monitor_on = on != 0;
    return 0;
}

extern "C" int sc_get_monitor(sc_ctx *ctx, double *sum_dv, int64_t *n) {
    CKR(enter(ctx, "sc_get_monitor"));
    if (!sum_dv) return fail(ctx, "sc_get_monitor: NULL argument");
    if (!ctx->monitor) return fail(ctx, "sc_get_monitor: sc_set_monitor(ctx, 1) has not been called");
    double h[8];
    CK(cudaMemcpyAsync(h, ctx->monitor, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    for (int q = 0; q < 6; ++q) sum_dv[q] = h[q];
    if (n) *n = (int64_t)h[6];
    return 0;
}

// ---- measurement -------------------------------------------------------------------------------------------
extern "C" int sc_profile_enable(sc_ctx *ctx, int on) {
    if (!ctx) return fail(ctx, "sc_profile_enable: NULL ctx");
    CK(cudaSetDevice(ctx->device));
    CKR(prof_flush(ctx));
    ctx->profiling = on != 0;
    if (on) for (int i = 0; i < SC_PROFILE_SLOTS; ++i) { ctx->prof_launches[i] = 0; ctx->prof_ms[i] = 0; }
    return 0;
}
extern "C" int sc_profile_read(sc_ctx *ctx, int64_t *launches, double *ms, int slots) {
    if (!ctx) return fail(ctx, "sc_profile_read: NULL ctx");
    CK(cudaSetDevice(ctx->device));
    CKR(prof_flush(ctx));
    for (int i = 0; i < slots && i < SC_PROFILE_SLOTS; ++i) {
        if (launches) launches[i] = ctx->prof_launches[i];
        if (ms) ms[i] = ctx->prof_ms[i];
    }
    return 0;
}
extern "C" const char *sc_profile_name(int slot) { return (slot >= 0 && slot < SC_PROFILE_SLOTS) ? k_slot_names[slot] : ""; }
extern "C" int64_t sc_launch_count(const sc_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" int64_t sc_sync_count(const sc_ctx *ctx) { return ctx ? ctx->syncs : 0; }


// ---- strip decomposition ------------------------------------------------------------------------------------
static int dist_ready(sc_ctx *ctx, const char *who) {
    CKR(require_ready(ctx, who));
    if (!ctx->dist_on) return fail(ctx, std::string(who) + ": sc_dist_configure has not been called");
    if (ctx->in_step) return fail(ctx, std::string(who) + ": inside a split step");
    return 0;
}

extern "C" int64_t sc_dist_wire_bytes(int64_t wire_capacity) {
    return (int64_t)sizeof(WireHeader) + (int64_t)sizeof(WireRec) * wire_capacity;
}

extern "C" int sc_dist_configure(sc_ctx *ctx, int rank, int nranks, int64_t row_lo, int64_t row_hi, int halo_rows,
                                 int64_t wire_capacity) {
    CKR(enter(ctx, "sc_dist_configure"));
    CKR(drop_keys(ctx));
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, "sc_dist_configure: bad rank");
    if (halo_rows < 1) return fail(ctx, "sc_dist_configure: halo_rows must be >= 1");
    if (wire_capacity < 1 || wire_capacity > ctx->cap) return fail(ctx, "sc_dist_configure: bad wire capacity");
    if (rank > 0 && rank < nranks - 1 && row_hi - row_lo < 2 * (int64_t)halo_rows)
        return fail(ctx, "sc_dist_configure: a strip must be at least 2 * halo_rows high");
    if (ctx->noise_mode == SC_NOISE_HOST) return fail(ctx, "sc_dist_configure: SC_NOISE_HOST is single-GPU only");
    ctx->dist.row_lo = row_lo; ctx->dist.row_hi = row_hi; ctx->dist.halo = halo_rows;
    ctx->dist.far_lo = row_lo - halo_rows; ctx->dist.far_hi = row_hi + halo_rows;  // until sc_dist_set_reach says more
    ctx->dist.reach_set = 0;
    ctx->dist.has_lo = rank > 0; ctx->dist.has_hi = rank < nranks - 1;
    ctx->dist.cap = (uint32_t)wire_capacity;
    if (!ctx->wire_dummy) {
        CKR(dev_alloc(ctx, &ctx->wire_dummy, 3));
        CK(cudaMemsetAsync(ctx->wire_dummy, 0, sizeof(WireHeader) * 3, ctx->stream));
    }
    ctx->dist_on = true;
    if (ctx->params_set) {
        CKR(sync_count(ctx));  // the live count may sit in the old cell array's tail
        CKR(world_grid(ctx));
    }
    return 0;
}

extern "C" int sc_dist_set_rows(sc_ctx *ctx, int64_t row_lo, int64_t row_hi) {
    CKR(dist_ready(ctx, "sc_dist_set_rows"));
    CKR(drop_keys(ctx));
    if (ctx->dist.has_lo && ctx->dist.has_hi && row_hi - row_lo < 2 * (int64_t)ctx->dist.halo)
        return fail(ctx, "sc_dist_set_rows: a strip must be at least 2 * halo_rows high");
    ctx->dist.row_lo = row_lo; ctx->dist.row_hi = row_hi;
    if (!ctx->dist.reach_set) { ctx->dist.far_lo = row_lo - ctx->dist.halo; ctx->dist.far_hi = row_hi + ctx->dist.halo; }
    // the restricted cell grid must still cover the strip, its halo and the wall-fix shift
    const long long need = ctx->dist.halo + 2;
    const long long g_lo = (long long)ctx->grid.row_min + 1, g_hi = (long long)ctx->grid.row_min + ctx->grid.nrows - 2;
    const bool lo_ok = !ctx->dist.has_lo || row_lo - need >= g_lo, hi_ok = !ctx->dist.has_hi || row_hi + need <= g_hi;
    if (!lo_ok || !hi_ok) {
        // the world grid is a superset check: rows of the world box are always inside (world_grid clamps to them)
        long long w_lo, w_hi;
        world_rows(ctx, w_lo, w_hi);
        if ((ctx->dist.has_lo && row_lo - need < g_lo && g_lo > w_lo) ||
            (ctx->dist.has_hi && row_hi + need > g_hi && g_hi < w_hi)) {
            CKR(sync_count(ctx));
            CKR(world_grid(ctx));
            ctx->n_host = ctx->cap;
            ctx->n_exact = false;
        }
    }
    return 0;
}

extern "C" int sc_dist_set_reach(sc_ctx *ctx, int64_t far_lo, int64_t far_hi) {
    CKR(dist_ready(ctx, "sc_dist_set_reach"));
    if (far_lo > ctx->dist.row_lo || far_hi < ctx->dist.row_hi) return fail(ctx, "sc_dist_set_reach: the reach must contain the strip");
    ctx->dist.far_lo = far_lo; ctx->dist.far_hi = far_hi; ctx->dist.reach_set = 1;
    return 0;
}

// weight of a particle in the re-cut histogram = work_base + its pair count (see k_dist_row_hist); SC_WORK_BASE overrides
static uint32_t work_base() {
    static int v = -1;
    if (v < 0) { const char *e = getenv("SC_WORK_BASE"); v = e ? atoi(e) : 2; if (v < 0) v = 0; }
    return (uint32_t)v;
}

extern "C" int sc_dist_row_histogram(sc_ctx *ctx, int64_t row0, int64_t nrows, uint64_t *hist) {
    CKR(dist_ready(ctx, "sc_dist_row_histogram"));
    if (nrows < 1 || nrows > (1 << 24) || !hist) return fail(ctx, "sc_dist_row_histogram: bad arguments");
    refresh_count(ctx);
    unsigned long long *d_hist = nullptr;
    CK(cudaMalloc((void **)&d_hist, sizeof(unsigned long long) * (size_t)nrows));
    CK(cudaMemsetAsync(d_hist, 0, sizeof(unsigned long long) * (size_t)nrows, ctx->stream));
    const int64_t n = ctx->n_host;
    // the particle arrays are still in the last tick's sorted order, whose pair counts are in pair_cnt
    const uint8_t *pc = ctx->rows_valid ? ctx->pair_cnt : nullptr;
    if (n > 0) {
        ProfScope ps(ctx, SLOT_IO);
        k_dist_row_hist<<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(&ctx->cnt->n, ctx->grid, ctx->pos_cur, ctx->uid_cur, pc,
                                                                     row0, (int)nrows, d_hist, work_base());
    }
    CK(cudaMemcpyAsync(hist, d_hist, sizeof(uint64_t) * (size_t)nrows, cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    CK(cudaFree(d_hist));
    return 0;
}

// pack (and, with peer pointers, push) the boundary particles of this tick
static int enqueue_pack(sc_ctx *ctx, const char *who, void *send_lo_dev, void *send_hi_dev, void *peer_recv_lo,
                        void *peer_flag_lo, void *peer_recv_hi, void *peer_flag_hi, bool direct, uint32_t value) {
    CKR(dist_ready(ctx, who));
    CKR(drop_keys(ctx));
    if ((ctx->dist.has_lo && !send_lo_dev) || (ctx->dist.has_hi && !send_hi_dev))
        return fail(ctx, std::string(who) + ": a neighbor exists but its send buffer is NULL");
    if (direct && ((ctx->dist.has_lo && (!peer_recv_lo || !peer_flag_lo)) || (ctx->dist.has_hi && (!peer_recv_hi || !peer_flag_hi))))
        return fail(ctx, std::string(who) + ": a neighbor exists but its peer pointers are NULL");
    WireHeader *lo = send_lo_dev ? (WireHeader *)send_lo_dev : ctx->wire_dummy;
    WireHeader *hi = send_hi_dev ? (WireHeader *)send_hi_dev : ctx->wire_dummy + 1;
    if (lo != ctx->send_lo || hi != ctx->send_hi) {  // first use of these buffers: arm them (later the pre-pass does)
        ProfScope ps(ctx, SLOT_IO);
        k_wire_reset<<<1, 1, 0, ctx->stream>>>(lo, hi);
        ctx->send_lo = lo; ctx->send_hi = hi;
    }
    // the live count: the previous tick's scan total if a step ran since cnt->n was last written
    const uint32_t *n_in = ctx->carry_count ? ctx->cell_start + ctx->grid.ncells : &ctx->cnt->n;
    ctx->carry_count = false;
    const int64_t n = ctx->n_host;
    const Grid &g = ctx->grid;
    // Boundary zones in sorted-index space (see k_dist_pack).  Rows that can hold a ghost, a migrant or a halo particle:
    // within halo of a cut, plus the rows a particle can cross in a tick (< 2) and a sliding cut can move (<= halo - 2),
    // on either side.  Valid only while the arrays are still in the order of the last search.
    PackRange R{nullptr, 0u, 0u};
    int64_t launch_n = n;
    if (ctx->rows_valid) {
        const long long zone = 2LL * ctx->dist.halo + 4;
        long long ra = ctx->dist.row_lo + zone - g.row_min, rb = ctx->dist.row_hi - zone - g.row_min;
        ra = ra < 0 ? 0 : (ra > g.nrows ? g.nrows : ra);
        rb = rb < 0 ? 0 : (rb > g.nrows ? g.nrows : rb);
        if (!ctx->dist.has_lo) ra = 0;
        if (!ctx->dist.has_hi) rb = g.nrows;
        if (ra < rb) {
            R.cell_start = ctx->cell_start;
            R.cell_a = (uint32_t)(ra * g.ncols); R.cell_b = (uint32_t)(rb * g.ncols);
            const int64_t zone_cap = 4LL * ctx->dist.cap;   // wire capacity is 4 (halo + 2) rows' worth: ample for two zones
            launch_n = std::min<int64_t>(n, zone_cap);
        }
    }
    PackOut plo{lo, reinterpret_cast<WireRec *>(lo + 1), nullptr, nullptr}, phi{hi, reinterpret_cast<WireRec *>(hi + 1), nullptr, nullptr};
    if (direct) {
        if (ctx->dist.has_lo) { plo.peer_hdr = (WireHeader *)peer_recv_lo; plo.recs = reinterpret_cast<WireRec *>(plo.peer_hdr + 1); plo.peer_flag = (uint32_t *)peer_flag_lo; }
        if (ctx->dist.has_hi) { phi.peer_hdr = (WireHeader *)peer_recv_hi; phi.recs = reinterpret_cast<WireRec *>(phi.peer_hdr + 1); phi.peer_flag = (uint32_t *)peer_flag_hi; }
    }
    uint32_t *done = &ctx->wire_dummy[2].count;  // "blocks done" counter of the direct kernel
    if (launch_n > 0) {
        ProfScope ps(ctx, SLOT_DIST_PACK);
        const dim3 grid(std::min<unsigned>(blocks_for(launch_n), 2 * 148)), block(SC_BLOCK);  // grid-stride: few, fat blocks
#define SC_PACK(REAL, DIRECT)                                                                                        \
        CK(launch_pdl(k_dist_pack<REAL, DIRECT>, grid, block, ctx->stream, ctx->cnt, n_in, g, ctx->dist, R,              \
                      ctx->pos_cur, (const Vec2<REAL>::type *)ctx->vel_cur, ctx->uid_cur, plo, phi, done, value))
        if (ctx->precision == SC_PRECISION_F64) { if (direct) SC_PACK(double, true); else SC_PACK(double, false); }
        else { if (direct) SC_PACK(float, true); else SC_PACK(float, false); }
#undef SC_PACK
    }
    CK(cudaGetLastError());
    ctx->srt_valid = false; ctx->rank_valid = false; ctx->lists_valid = false; ctx->rows_valid = false;
    ctx->n_exact = false;
    return 0;
}

extern "C" int sc_dist_pack(sc_ctx *ctx, void *send_lo_dev, void *send_hi_dev) {
    return enqueue_pack(ctx, "sc_dist_pack", send_lo_dev, send_hi_dev, nullptr, nullptr, nullptr, nullptr, false, 0u);
}

extern "C" int sc_dist_pack_push(sc_ctx *ctx, void *send_lo_dev, void *peer_recv_lo_dev, void *peer_flag_lo_dev,
                                 void *send_hi_dev, void *peer_recv_hi_dev, void *peer_flag_hi_dev, uint32_t value) {
    return enqueue_pack(ctx, "sc_dist_pack_push", send_lo_dev, send_hi_dev, peer_recv_lo_dev, peer_flag_lo_dev,
                        peer_recv_hi_dev, peer_flag_hi_dev, true, value);
}

// The unpack is only recorded: the next step's pre-pass appends the records (PrepassUnpack) and enter() holds every
// other call off until then.
static int record_unpack(sc_ctx *ctx, const void *recv_lo, const void *flag_lo, const void *recv_hi, const void *flag_hi,
                         uint32_t value) {
    CKR(drop_keys(ctx));
    ctx->pend.on = true;
    ctx->pend.recv_lo = recv_lo; ctx->pend.flag_lo = flag_lo; ctx->pend.recv_hi = recv_hi; ctx->pend.flag_hi = flag_hi;
    ctx->pend.value = value;
    // the live count (owned + ghosts) is only known on the device: launch over the whole capacity, kernels exit early
    ctx->n_host = ctx->cap;
    ctx->n_exact = false;
    return 0;
}

extern "C" int sc_dist_unpack(sc_ctx *ctx, const void *recv_lo_dev, const void *recv_hi_dev) {
    CKR(dist_ready(ctx, "sc_dist_unpack"));
    return record_unpack(ctx, recv_lo_dev, nullptr, recv_hi_dev, nullptr, 0);
}

extern "C" int sc_dist_unpack_flagged(sc_ctx *ctx, const void *recv_lo_dev, const void *flag_lo_dev,
                                      const void *recv_hi_dev, const void *flag_hi_dev, uint32_t value) {
    CKR(dist_ready(ctx, "sc_dist_unpack_flagged"));
    return record_unpack(ctx, recv_lo_dev, flag_lo_dev, recv_hi_dev, flag_hi_dev, value);
}

// NOTE: the unpacking pre-pass clamps the appended count on overflow only by flagging; cnt->n may exceed cap by the
// number of dropped records, every kernel bounds its index by the arrays' capacity through n_host <= cap.
extern "C" int sc_dist_get_owned(sc_ctx *ctx, double *pos, double *vel, uint32_t *uid, int64_t cap, int64_t *n_out) {
    CKR(dist_ready(ctx, "sc_dist_get_owned"));
    refresh_count(ctx);
    CK(cudaMemsetAsync(&ctx->cnt->n_tmp, 0, sizeof(uint32_t), ctx->stream));
    const int64_t n = ctx->n_host;
    if (n > 0) {
        ProfScope ps(ctx, SLOT_IO);
        if (ctx->precision == SC_PRECISION_F64)
            k_dist_collect_owned<double><<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(
                &ctx->cnt->n, ctx->pos_cur, (const double2 *)ctx->vel_cur, ctx->uid_cur, ctx->stage2, ctx->pos_srt,
                (uint32_t *)ctx->stage1, &ctx->cnt->n_tmp);
        else
            k_dist_collect_owned<float><<<blocks_for(n), SC_BLOCK, 0, ctx->stream>>>(
                &ctx->cnt->n, ctx->pos_cur, (const float2 *)ctx->vel_cur, ctx->uid_cur, ctx->stage2, ctx->pos_srt,
                (uint32_t *)ctx->stage1, &ctx->cnt->n_tmp);
    }
    ctx->srt_valid = false;
    Counters h;
    CK(cudaMemcpyAsync(&h, ctx->cnt, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    if (n_out) *n_out = h.n_tmp;
    if ((int64_t)h.n_tmp > cap) return fail(ctx, "sc_dist_get_owned: buffer too small");
    const size_t m = h.n_tmp;
    if (m && pos) CK(cudaMemcpyAsync(pos, ctx->stage2, sizeof(double2) * m, cudaMemcpyDeviceToHost, ctx->stream));
    if (m && vel) CK(cudaMemcpyAsync(vel, ctx->pos_srt, sizeof(double2) * m, cudaMemcpyDeviceToHost, ctx->stream));
    if (m && uid) CK(cudaMemcpyAsync(uid, ctx->stage1, sizeof(uint32_t) * m, cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    return 0;
}

// flags raised on the device since the context was created: wire / particle capacity overflow, a particle that
// moved past a whole halo in one tick.  `send_*_dev` may be NULL.  Synchronises.
extern "C" int sc_dist_status(sc_ctx *ctx, const void *send_lo_dev, const void *send_hi_dev, int *overflow,
                              int *too_far, int64_t *n_local) {
    CKR(dist_ready(ctx, "sc_dist_status"));
    CKR(sync_count(ctx));
    Counters h;
    CK(cudaMemcpyAsync(&h, ctx->cnt, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
    WireHeader w[2] = {};
    if (send_lo_dev && ctx->dist.has_lo) CK(cudaMemcpyAsync(&w[0], send_lo_dev, sizeof(WireHeader), cudaMemcpyDeviceToHost, ctx->stream));
    if (send_hi_dev && ctx->dist.has_hi) CK(cudaMemcpyAsync(&w[1], send_hi_dev, sizeof(WireHeader), cudaMemcpyDeviceToHost, ctx->stream));
    CK(stream_sync(ctx));
    if (overflow) *overflow = (h.overflow || w[0].overflow || w[1].overflow || h.n > (uint32_t)ctx->cap) ? 1 : 0;
    if (too_far) *too_far = (w[0].too_far || w[1].too_far) ? 1 : 0;
    if (n_local) *n_local = h.n;
    ctx->n_host = ctx->cap;  // back to the conservative launch bound (sync_count narrowed it)
    ctx->n_exact = false;
    return 0;
}
