/*
 * sandcrate.h - C ABI of the B200 (sm_100a) implementation of SandCrate's per-timestep particle step.
 *
 * The reference (David-Taub/sand_crate) has no FFI: its step is the Python method `Crate.physics_tick()`
 * (src/crate/crate.py:91-129).  This header is the boundary a maintainer binds instead (ctypes stub in
 * INTEGRATION.md; the in-repo binding is sand_crate_b200/_lib.py).  Each entry point cites the reference
 * code it replaces.  Plain pointers and sizes only; every `const double*` / `double*` is a HOST pointer borrowed
 * for the duration of the call unless the name says `_dev`.
 *
 * Conventions
 *   - return value: 0 = ok, non-zero = error; `sc_last_error(ctx)` (or `sc_last_error(NULL)` for `sc_create`)
 *     returns the message.  CUDA errors are reported, never swallowed; there is no CPU fallback.
 *   - one context per GPU, not thread-safe, all work on one CUDA stream.
 *   - particles keep their identity (a stable 32-bit uid = order of insertion); every host-visible per-particle
 *     array is in the reference's "original index" order (ascending uid among live particles), exactly like
 *     the rows of `Crate.particles` (crate.py:24, 146-159).
 */
#ifndef SANDCRATE_H
#define SANDCRATE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SC_MAX_NEIGHBORS 20 /* collision_detector.py:6 MAX_ALLOWED_NEIGHBORS */
#define SC_MAX_SEGMENTS 32  /* wall segments per scene (stirring_cup: 6, wave_machine: 8) */
#define SC_MAX_BODIES 16

typedef struct sc_ctx sc_ctx;

/* world.coefficients of config/*.yaml (stirring_cup.yaml:9-22), the ones the step reads (crate.py:42-57).
 * spring_overlap_balance / spring_amplifier are dead in the reference (crate.py:117-118) and max_particles is a
 * host-side source limit, so they are not part of the device parameter block. */
typedef struct sc_params {
    double dt;
    double particle_radius;
    double wall_collision_decay;
    double pressure_amplifier;
    double ignored_pressure;
    double collider_noise_level;
    double viscosity;
    double surface_smoothing;
    double target_pressure;
    double gravity_x;
    double gravity_y;
} sc_params;

/* arithmetic mode of the pair / force kernels */
#define SC_PRECISION_F64 0   /* fp64, no FMA contraction, reference summation orders: bit-exact parity mode */
#define SC_PRECISION_MIXED 1 /* positions fp64 in HBM, pair differences fp64 -> fp32, forces/velocities fp32 */

/* source of the per-directed-pair collider noise (crate.py:168-170) */
#define SC_NOISE_NONE 0    /* term skipped; exact when collider_noise_level == 0 */
#define SC_NOISE_COUNTER 1 /* counter-based: lowbias32(uid_i * C1 ^ uid_j * C2 ^ fold32(tick_key(seed, tick))), 2 x 16 bits */
#define SC_NOISE_HOST 2    /* the caller supplies the reference's own np.random.rand stream per tick */

/* ---- lifetime ------------------------------------------------------------------------------------------ */
/* `stream` is a cudaStream_t the caller owns (e.g. torch.cuda.current_stream().cuda_stream) or NULL for a
 * private stream.  `capacity` = maximum number of live particles (crate.py `max_particles`). */
int sc_create(int device, int precision, int64_t capacity, void *stream, sc_ctx **out);
void sc_destroy(sc_ctx *ctx);
const char *sc_last_error(const sc_ctx *ctx);
int sc_version(void);

/* ---- configuration (re-read every tick by the reference: playback.py:221-226 edits coefficients live) --- */
int sc_set_params(sc_ctx *ctx, const sc_params *p);                 /* crate.py:55-57 */
/* segments: S x 4 (ax, ay, bx, by) = `Crate.segments` (crate.py:69-71) AFTER apply_bodies_velocity
 * (crate.py:363-365); body_len[nbodies] = segments per body; body_kin: nbodies x 5 =
 * (center_velocity.x, .y, angular_clockwise_velocity, position.x, .y) (rigid_body.py:18-34). */
int sc_set_walls(sc_ctx *ctx, const double *segments, int S, const int32_t *body_len, const double *body_kin,
                 int nbodies);
int sc_set_noise(sc_ctx *ctx, int mode, uint64_t seed);
int sc_set_tick(sc_ctx *ctx, uint64_t tick);                        /* crate.py:23, 127 */

/* ---- state ------------------------------------------------------------------------------------------- */
int sc_set_state(sc_ctx *ctx, const double *pos, const double *vel, int64_t n); /* uid = 0..n-1 */
/* create_new_particles (crate.py:138-147): appended rows get the next uids. */
int sc_append_particles(sc_ctx *ctx, const double *pos, const double *vel, int64_t n);
int sc_particle_count(sc_ctx *ctx, int64_t *n);                     /* crate.py:87-89; synchronises */
/* any of pos / vel / pressure may be NULL.  pos, vel: n x 2; pressure: n (crate.py:26, 275). */
int sc_get_state(sc_ctx *ctx, double *pos, double *vel, double *pressure, int64_t cap, int64_t *n);
int sc_get_uids(sc_ctx *ctx, uint32_t *uid, int64_t cap, int64_t *n);
/* The uid the next appended or emitted particle gets (identities advance by the drawn count, so a clamped emission
 * leaves a gap that sc_set_state_uids alone cannot restore).  Refused below the context's current next uid and at or
 * above 2^31.  With sc_set_state_uids it moves a scene into a new context with its identities intact. */
int sc_set_next_uid(sc_ctx *ctx, uint32_t next_uid);

/* Between ticks.  A call that returns an error leaves the context as it was.  Readbacks (sc_get_state, sc_get_uids,
 * sc_particle_count), the parity taps, the diagnostics, measurement, the ForceMonitor switch, sc_synchronize and a
 * configuration call with the bytes already set (sc_set_params, sc_set_walls, sc_set_tick) never change a later result.
 * Pressure reads as the last tick computed it for each particle, and 0 for every particle once sc_set_state,
 * sc_set_state_uids, sc_append_particles or sc_emit_particles changed the particle set since (crate.py:26); a re-grid (a
 * new particle_radius, or walls that need more wall-contact room) keeps it, though the parity taps then refuse until the
 * next step.  Inside a split step (between sc_step_begin and sc_step_finish) the parity taps but sc_get_tension,
 * sc_set_params without a radius change, sc_set_noise, sc_set_tick, sc_set_walls with the walls already set,
 * sc_last_pair_count, sc_synchronize and measurement are allowed; sc_get_state, sc_get_uids, sc_set_state,
 * sc_append_particles, sc_emit_particles, sc_step, a radius change and a change of walls are refused. */

/* create_new_particles + ParticleSource.generate_particles (crate.py:138-147, particle_source.py:17-24) on the DEVICE,
 * for the counter-based production mode (the reference-stream mode keeps drawing on the host and appends with
 * sc_append_particles).  `count` = the emission count the caller drew for this tick from the counter stream
 * (sc_source_stream element 0 through the binomial inverse CDF: sand_crate_b200/particle_source.py); the device clamps
 * it to max_particles - particle_count exactly where the reference does (count before this tick's removal, after the
 * earlier sources), draws positions / velocities from stream elements 1 + 4k + {0, 1, 2, 3} and appends.  No host
 * synchronisation: a tick with sources costs one extra one-block launch.  Uses the seed of sc_set_noise and the tick
 * of sc_set_tick. */
typedef struct sc_source {
    double position_x, position_y; /* ParticleSource.position */
    double radius;                 /* .radius */
    double velocity_x, velocity_y; /* .velocity */
    double velocity_noise;         /* .noise */
    int32_t count;                 /* drawn emission count of this tick */
    uint32_t index;                /* position of the source in world.particle_sources (keys its stream) */
} sc_source;
#define SC_MAX_SOURCES 8
int sc_emit_particles(sc_ctx *ctx, const sc_source *sources, int nsources, int64_t max_particles);
/* element j of source `source_index`'s counter stream at (seed, tick) as a uniform in [0, 1); returns the stream key */
uint64_t sc_source_stream(uint64_t seed, uint64_t tick, uint32_t source_index, uint64_t j, double *u);

/* Page-locked host memory for the buffers handed to sc_set_state / sc_append_particles / sc_get_state /
 * sc_dist_get_owned.  No reference counterpart (the reference never leaves the host); with pageable buffers the
 * copies are staged by the driver and run at a fraction of the PCIe rate.  The host mirror keeps its readback arrays
 * (crate.py:24-26 `particles`, `particle_velocities`, `particles_pressure`) in such memory. */
int sc_host_alloc(size_t bytes, void **out);
int sc_host_free(void *p);

/* ---- the step ------------------------------------------------------------------------------------------ */
/* One tick = remove_particles (crate.py:149-159) -> calc_virtual_colliders + apply_hard_wall_fix (213-243,
 * 202-211) -> detect_particle_collisions (collision_detector.py:9-49) -> populate_colliders (161-175) ->
 * pressures (261-284) -> tension, gravity, pressure, viscosity (335-353, 309-310, 295-307, 316-323) ->
 * wall bounce (245-259) -> continuous collision (177-200) -> integration (360-361); tick += 1.
 * Asynchronous: returns after enqueueing.  Not valid with SC_NOISE_HOST (use begin/finish). */
int sc_step(sc_ctx *ctx);
int sc_step_n(sc_ctx *ctx, int nsteps);
/* Split form for SC_NOISE_HOST: `begin` runs everything up to and including the neighbor search and returns
 * the live particle count and the number of directed pairs sum(K_i); the caller draws `n_pairs x 2` uniforms
 * from the reference's generator (CSR order: particle ascending, slot ascending, x then y - crate.py:165-170)
 * and passes them to `finish`.  With other noise modes `noise` is ignored. */
int sc_step_begin(sc_ctx *ctx, int64_t *n_particles, int64_t *n_pairs);
int sc_step_finish(sc_ctx *ctx, const double *noise);
int sc_synchronize(sc_ctx *ctx);

/* ---- parity taps (valid after sc_step / sc_step_begin; all in original index order) -------------------- */
/* pos_search: positions the search ran on (after apply_hard_wall_fix); rows_sorted / order:
 * `y_floored[sorted_indices]`, `sorted_indices` of strip_sort_particles (collision_detector.py:124-128). */
int sc_get_search(sc_ctx *ctx, double *pos_search, int64_t *rows_sorted, int64_t *order, int64_t cap);
/* `colliders_indices` (crate.py:102): counts[n], idx[n x 20] holding original indices, -1 padded. */
int sc_get_neighbors(sc_ctx *ctx, int32_t *counts, int32_t *idx, int64_t cap);
/* surface normals of apply_tension pass 1 (crate.py:337-342), n x 2. */
int sc_get_tension(sc_ctx *ctx, double *tension, int64_t cap);
/* number of wall contacts V_i per particle (crate.py:229-232) of the last tick. */
int sc_get_wall_counts(sc_ctx *ctx, int32_t *counts, int64_t cap);

/* ---- the reference's layer-2 functions as standalone device ops ---------------------------------------- */
/* detect_particle_collisions(particles, diameter) (collision_detector.py:9-49) on arbitrary coordinates. */
int sc_detect_particle_collisions(sc_ctx *ctx, const double *particles, int64_t P, double diameter,
                                  int64_t *rows_sorted, int64_t *order, int32_t *counts, int32_t *idx);
/* points_to_segments_distance (geometry_utils.py:7-39): nearest P x S x 2, dist P x S. */
int sc_points_to_segments_distance(sc_ctx *ctx, const double *p, int64_t P, const double *segments, int S,
                                   double *nearest, double *dist);
/* pad_segments (geometry_utils.py:146-172): padded 2S x 4. */
int sc_pad_segments(const double *segments, int S, double pad, double *padded);

/* ---- ForceMonitor (utils/force_monitor.py:13-37) -------------------------------------------------------------- */
/* With the monitor on, every tick also sums |dv| over the particles for each of the six sections the reference
 * wraps in `force_monitor(...)` (crate.py:110-124): tension, gravity, pressure, viscosity, wall_bounce,
 * continuous_collision.  sc_get_monitor returns the six sums and the particle count of the last tick; the mean and
 * the reference's 0.8 decay are the caller's (sand_crate_b200/crate.py).  Synchronises. */
int sc_set_monitor(sc_ctx *ctx, int on);
int sc_get_monitor(sc_ctx *ctx, double *sum_dv, int64_t *n);

/* ---- measurement ---------------------------------------------------------------------------------------- */
/* Per-kernel CUDA-event timing on the context's stream.  sc_profile_read returns, for each kernel slot, the
 * number of launches and the summed milliseconds since sc_profile_enable(ctx, 1). */
#define SC_PROFILE_SLOTS 16
int sc_profile_enable(sc_ctx *ctx, int on);
int sc_profile_read(sc_ctx *ctx, int64_t *launches, double *ms, int slots);
const char *sc_profile_name(int slot);
int64_t sc_launch_count(const sc_ctx *ctx); /* kernels launched by this context so far */
int64_t sc_sync_count(const sc_ctx *ctx);   /* times an entry point made the host wait for the stream so far */
/* sum(K_i) of the last tick = rows of the reference's `colliders` lists (crate.py:161-175) over the particles this
 * context holds (ghost copies of a strip included).  Synchronises. */
int sc_last_pair_count(sc_ctx *ctx, int64_t *n_pairs);

/* ---- diagnostics (developer aids; no reference counterpart, results are never affected) ---------------------- */
/* re-run the density (which = 4) or force (which = 5) kernel of the last tick `reps` times; mean milliseconds.
 * -1 before a step, inside a split step, under SC_NOISE_HOST (the step's noise offsets do not outlive it) and once a
 * call has changed the parameters, walls or noise the step ran with.  The re-run takes back the next tick's keys (that
 * tick then runs its own pre-pass), like every call that touches what they depend on. */
double sc_debug_rerun(sc_ctx *ctx, int which, int reps);
/* blocks of the tiled density kernel that ran in pass-through mode in the last tick (windows too large to stage) */
int64_t sc_debug_untiled_blocks(sc_ctx *ctx);
/* The pair records the density kernel of the last tick handed to its force kernel, in original index order:
 * counts[n] = K_i as stored, nbr_row[n x 20] = the neighbors' original indices in list order (-1 padded),
 * nvec[n x 20 x 2] = the unit vectors as the force kernel decodes them (fp32 in mixed precision, widened).  Valid from
 * the end of sc_step / sc_step_finish until the next step or sc_debug_rerun rewrites the pair buffers; refused inside a
 * split step (the buffers still hold the tick before).  Synchronises. */
int sc_debug_pair_records(sc_ctx *ctx, int32_t *counts, int32_t *nbr_row, double *nvec, int64_t cap);
/* the cell grid: grid4 = {row_min, col_min, nrows, ncols}; cell of (row, col) = (row - row_min) * ncols + col - col_min,
 * both clamped to [1, size - 2] */
int sc_debug_grid(sc_ctx *ctx, int64_t *grid4);
/* The conservative wall culls of the current walls (never change a result, only skip work), each box / rectangle as
 * (xmin, xmax, ymin, ymax): rects[12] = safe_contact, safe_ccd, safe_ccd_f32 (widened to double); seg_box[S x 4] =
 * each segment's box grown by the touch distance; pad_box[2S x 4] = each padded segment's box.  Buffers may be NULL;
 * the boxes need room for SC_MAX_SEGMENTS rows.  counts[2] = {S, the wall contacts per particle the cell grid has room
 * for}.  Refused before sc_set_walls. */
int sc_debug_walls(sc_ctx *ctx, double *rects, double *seg_box, double *pad_box, int32_t *counts);

/* ---- multi-GPU strip decomposition (one context per rank) ------------------------------------------------------ */
/* The reference's search is already a 1-D strip decomposition in y with strip height one diameter
 * (collision_detector.py:10-31, 124-128); rank k owns the cell rows row_lo <= floor(y / d) < row_hi.  Every tick,
 * before sc_step, one of two transports:
 *   caller's send/recv   sc_dist_pack -> the caller exchanges the buffers, whole, with rank - 1 / rank + 1 (e.g. NCCL)
 *                        -> sc_dist_unpack
 *   direct (NVLink)      sc_dist_pack_push -> sc_dist_unpack_flagged
 * The pack drops last tick's ghosts, turns particles whose row left the strip into MIGRANT records for the neighbor
 * (they stay here as ghosts for this tick) and copies owned particles within `halo_rows` of a cut into HALO records;
 * send_*_dev: device buffers of sc_dist_wire_bytes(capacity) bytes (16-byte header with the record count, then 40-byte
 * records), NULL where there is no neighbor.  The unpack appends received migrants as owned particles and received
 * halos as ghosts.  A ghost is simulated like any particle and discarded by the next pack.  With the halo the walls
 * need (sc_dist_halo_rows: 2 + 2 ceil(V r / d) rows for walls that give a particle up to V contacts, 4 for V <= 2)
 * every owned particle sees the neighbors, pressures and normals of the global computation in the same order:
 * results are bit-identical to a single-GPU run.  sc_dist_configure, and sc_set_walls on a strip context, refuse
 * walls that need more halo rows than configured (nothing is launched, the message names the halo needed).
 * The unpack only records the receive buffers: the next step's first kernel appends their records.  Until then the
 * particle state is incomplete, so the next call on the context must be sc_step, sc_step_n or sc_step_begin; only
 * sc_set_tick, sc_synchronize, sc_destroy, sc_last_error, sc_profile_*, sc_launch_count and sc_sync_count may come
 * before it.  Every other call that takes the context returns an error.
 * Restrictions of the strip mode: noise must be SC_NOISE_COUNTER or SC_NOISE_NONE (the reference's global RNG
 * stream cannot be split across ranks); uids must be < 2^31 (bit 31 marks a ghost copy); particle sources go through
 * sc_dist_emit_particles (sc_emit_particles is refused); on a context with a neighbor, sc_get_state / sc_get_uids /
 * the parity taps return an error - read back with sc_dist_get_owned.  Moving bodies need nothing special: every
 * rank passes the same walls to sc_set_walls. */
int64_t sc_dist_wire_bytes(int64_t wire_capacity);
int sc_dist_configure(sc_ctx *ctx, int rank, int nranks, int64_t row_lo, int64_t row_hi, int halo_rows,
                      int64_t wire_capacity);
int sc_dist_pack(sc_ctx *ctx, void *send_lo_dev, void *send_hi_dev);
int sc_dist_unpack(sc_ctx *ctx, const void *recv_lo_dev, const void *recv_hi_dev);
/* The direct transport.  sc_dist_pack_push is sc_dist_pack whose records are written straight into the neighbors'
 * receive buffers through peer-mapped device pointers (e.g. torch symmetric memory) as they are produced; the last
 * block to finish publishes the counts and stores `value` (release, system scope) to each neighbor's flag word.
 * send_*_dev are still needed (their headers hold the record counters and the sticky overflow / too_far marks).
 * sc_dist_unpack_flagged is sc_dist_unpack whose records are read (on the device) only once this rank's flag words
 * have reached `value`.  Use the tick number as `value`: monotonic, never reset.  NULL where there is no neighbor. */
int sc_dist_pack_push(sc_ctx *ctx, void *send_lo_dev, void *peer_recv_lo_dev, void *peer_flag_lo_dev, void *send_hi_dev,
                      void *peer_recv_hi_dev, void *peer_flag_hi_dev, uint32_t value);
int sc_dist_unpack_flagged(sc_ctx *ctx, const void *recv_lo_dev, const void *flag_lo_dev, const void *recv_hi_dev,
                           const void *flag_hi_dev, uint32_t value);
/* owned particles of this rank, in arbitrary order; uid[i] identifies row i.  Synchronises. */
int sc_dist_get_owned(sc_ctx *ctx, double *pos, double *vel, uint32_t *uid, int64_t cap, int64_t *n);
/* device-side flags since creation: capacity overflow, a particle that crossed a whole halo in one tick; the
 * number of local particles (owned + ghosts).  Synchronises. */
int sc_dist_status(sc_ctx *ctx, const void *send_lo_dev, const void *send_hi_dev, int *overflow, int *too_far,
                   int64_t *n_local);
/* Re-balancing the partition.  sc_dist_row_histogram: WORK of the owned particles per cell row (2 + the particle's
 * pair count of the last tick; equal weights before the first tick), rows row0 .. row0 + nrows - 1 (outliers clamped to the
 * ends); the caller sums it over the ranks (the only collective of the scheme, on
 * re-cut ticks only) and derives new cuts.  sc_dist_set_rows moves this rank's cuts; a cut may move by less than
 * `halo_rows` rows per tick - the rows it hands over then travel as ordinary migrants of the next sc_dist_pack. */
int sc_dist_row_histogram(sc_ctx *ctx, int64_t row0, int64_t nrows, uint64_t *hist);
int sc_dist_set_rows(sc_ctx *ctx, int64_t row_lo, int64_t row_hi);
/* How far a migrant may land: far_lo / far_hi = the first row of the lower neighbor's strip / one past the last row of
 * the upper neighbor's.  A particle that crosses a cut is handed to the adjacent rank only, so it must land inside that
 * rank's strip; beyond it the too_far flag is raised.  Default reach: halo_rows past the cut (the round-1 rule), which
 * is tighter than necessary - the wall jets of a 8 000-row dam break move 3 rows per tick.  Call again after
 * sc_dist_set_rows when the neighbors' cuts move. */
int sc_dist_set_reach(sc_ctx *ctx, int64_t far_lo, int64_t far_hi);
/* like sc_set_state but with caller-chosen uids (global particle ids of a partitioned scene) */
int sc_set_state_uids(sc_ctx *ctx, const double *pos, const double *vel, const uint32_t *uid, int64_t n);
/* The halo rows a strip needs under walls `segments` (S x 4, as sc_set_walls) for particles of radius
 * `particle_radius` (see above); -1 for bad arguments.  Host arithmetic, no context. */
int sc_dist_halo_rows(const double *segments, int S, double particle_radius);
/* Particle sources on a strip.  sc_dist_owned_count enqueues a kernel that writes this rank's live particles that are
 * not ghosts to the caller's device word `count_dev` (no host wait); summed over the ranks (e.g. an all-reduce on the
 * context's stream) it is the scene's particle_count that sc_emit_particles clamps against.  Take it before
 * sc_dist_pack: last tick's ghosts are excluded and a particle about to migrate is counted once.
 * sc_dist_emit_particles is sc_emit_particles for a strip: every rank passes the same records, the same
 * `max_particles` and the same scene-wide `first_uid` (the uid of the tick's first drawn particle; identities advance by
 * the drawn counts, so the caller tracks it without device data).  The device clamps each source exactly like
 * sc_emit_particles with particle_count read from `scene_count_dev` (NULL: the caller has proven that the clamp cannot
 * bind, every drawn particle is emitted), generates the same stream elements and identities, and appends only the
 * particles whose row floor(y / d) this rank owns, in (source, particle) order.  The next sc_dist_pack sends the ones
 * within a halo of a cut to the neighbor.  A rank whose capacity is exceeded raises the overflow flag. */
int sc_dist_owned_count(sc_ctx *ctx, uint32_t *count_dev);
int sc_dist_emit_particles(sc_ctx *ctx, const sc_source *sources, int nsources, int64_t max_particles,
                           uint32_t first_uid, const uint32_t *scene_count_dev);

/* ---- ensembles: M members of one scene in one context (DESIGN.md section 12) ------------------------------------ */
/* An ensemble steps M variants of one scene - a coefficient sweep or seed replicas - with one launch sequence per tick
 * whatever M is.  The members share dt, particle_radius and the walls (sc_set_walls, once for all); each has its own
 * other coefficients, noise seed, particles and identities, and each is bit-identical to a single-scene context run with
 * its coefficients and seed.  Member m's cells are m * (cells of the scene's grid) + its own cell, so the cell grid is
 * the scene's stacked M times and M times its cells must fit the 32-bit cell key; member m's uids are
 * (m << uid_bits) | local uid, local uids in order of creation as on a single-scene context.
 * sc_ens_configure makes a fresh context (no parameters, no state yet) an ensemble.  M * 2^uid_bits <= 2^31; the
 * readback map takes 4 * M * 2^uid_bits bytes of device memory.  Refused with SC_NOISE_HOST, on a strip context and with
 * the ForceMonitor on; those calls are refused on an ensemble later as well.
 * On an ensemble context:
 *   works, all members at once: sc_set_walls, sc_set_tick, sc_step, sc_step_n, sc_synchronize, sc_particle_count (the
 *     total), sc_get_state / sc_get_uids (all members, member-major = ascending global uid; the uids are global),
 *     sc_last_pair_count (the directed pairs of all members), measurement, sc_debug_untiled_blocks, sc_debug_grid (the
 *     stacked grid), sc_debug_walls, sc_detect_particle_collisions / sc_points_to_segments_distance (they do not touch
 *     the context's state);
 *   sc_set_noise: the mode only (SC_NOISE_COUNTER or SC_NOISE_NONE); the seeds come with sc_ens_set_params;
 *   refused: sc_set_params, sc_set_state, sc_set_state_uids, sc_append_particles, sc_emit_particles (use the sc_ens_
 *     forms), sc_step_begin / sc_step_finish, the parity taps, sc_debug_pair_records, sc_debug_rerun (returns -1),
 *     sc_set_monitor and sc_get_monitor (the monitor cannot be switched on, so there is nothing to read), sc_set_state_uids,
 *     sc_set_next_uid,
 *     sc_dist_* (sc_dist_configure refuses; the other sc_dist_ calls need it). */
int sc_ens_configure(sc_ctx *ctx, int members, int uid_bits);
/* p[M], seeds[M]: each member's coefficients and noise seed.  dt and particle_radius must be the same in every member
 * (the error names the field and the member).  Changing any member's bytes drops the next tick's precomputed keys, as
 * sc_set_params does; pushing unchanged bytes costs no launch. */
int sc_ens_set_params(sc_ctx *ctx, const sc_params *p, const uint64_t *seeds);
/* The whole state: pos, vel = n x 2 with n = sum(counts), member 0's rows first.  uid[n]: the rows' global uids (each
 * one of its member's), or NULL for local uids 0 .. counts[m] - 1; next_local[M]: the local uid each member's next
 * particle gets, or NULL for one past its largest.  (With both, a state read back with sc_ens_get_state and sc_get_uids
 * continues exactly in a context of another capacity.) */
int sc_ens_set_state(sc_ctx *ctx, const double *pos, const double *vel, const int64_t *counts, const uint32_t *uid,
                     const uint32_t *next_local);
/* sc_emit_particles for every member: sources[nsources] as for sc_emit_particles (their `count` is ignored),
 * counts[M x nsources] = the counts member m drew from its own counter stream (its seed), max_particles[M].  Each member
 * is clamped against its own live count, and its identities advance by its drawn count.  The draws travel as kernel
 * parameters: one launch while M * (nsources + 1) <= 7936, one more per further 7936 words.  No host wait, no host
 * buffer copied.  Refused before anything is launched when a member's identities would pass 2^uid_bits, and when the
 * members' counts could outgrow the capacity: each member's count is bounded by what the last state set and what every
 * emission's clamp allowed since (max(bound, min(bound + drawn, max_particles))), and the sum must fit. */
int sc_ens_emit_particles(sc_ctx *ctx, const sc_source *sources, int nsources, const int32_t *counts,
                          const int64_t *max_particles);
/* Per-member live counts: to the caller's device words counts_dev[M] (uint32, may be NULL; enqueued, no host wait) and,
 * when counts[M] is not NULL, to the host (synchronises). */
int sc_ens_member_counts(sc_ctx *ctx, int64_t *counts, uint32_t *counts_dev);
/* sc_get_state of all members, member-major, with offsets[M + 1]: member m's rows are offsets[m] .. offsets[m + 1] - 1.
 * Synchronises. */
int sc_ens_get_state(sc_ctx *ctx, double *pos, double *vel, double *pressure, int64_t cap, int64_t *offsets);

#ifdef __cplusplus
}
#endif
#endif /* SANDCRATE_H */
