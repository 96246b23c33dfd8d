/*
 * drstencil.h -- C ABI of the B200-native stencil engine (libdrstencil.so).
 *
 * The reference (simple86/DRStencil) has no library boundary: its "API" is the generator CLI
 * (/root/reference/main.cpp:10-280), the text of the emitted .cu (codegen_2d.hpp:49-75,
 * codegen.hpp:47-71) with the kernel `__global__ void dr_<name>(double*, double*)`
 * (codegen_2d.hpp:154,461; codegen.hpp:148) and the host loop the emitted main() runs around it
 * (codegen_2d.hpp:564-664; codegen.hpp:547-635).  Each entry point below names the piece of
 * that flow it stands in for.  Plain pointers and sizes only; every function returns 0 on
 * success or a negative DRS_E_* code and never calls exit(); drs_last_error() gives the text.
 *
 * Threading: a drs_stencil / drs_plan may be used by one host thread at a time; different
 * objects are independent.  Device buffers are caller-owned (any allocator: cudaMalloc, torch).
 */
#ifndef DRSTENCIL_H_
#define DRSTENCIL_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRS_OK 0
#define DRS_E_ARG (-1)        /* bad argument / unsupported description                        */
#define DRS_E_IO (-2)         /* .stc unreadable (reference: "Error opening stencil file.", rc 255) */
#define DRS_E_NOREUSE (-3)    /* reference: "No data to reuse. You can try another dist.", rc 1    */
#define DRS_E_CONFIG (-4)     /* reference: "Invalid configuration!", rc 255                     */
#define DRS_E_COMPILE (-5)    /* kernel specialisation failed (NVRTC log in drs_last_error)      */
#define DRS_E_CUDA (-6)       /* CUDA driver/runtime error                                      */
#define DRS_E_NOGPU (-7)      /* no usable CUDA device: the engine has NO CPU fallback          */
#define DRS_E_KERNEL (-8)     /* kernel reported an internal fault (pipeline watchdog)          */

#define DRS_F64 0
#define DRS_F32 1             /* extension: the reference is fp64 only                          */

#define DRS_FUSE_TEMPORAL 0   /* --step n = n in-kernel sub-steps of the base operator          */
#define DRS_FUSE_ALGEBRAIC 1  /* --step n = the composed (fused) operator evaluated literally,   */
                              /*            exactly what the reference emits                    */
#define DRS_FUSE_REUSE 2      /* A/B mode: the composed operator through the reference's forward / */
                              /* backward data-reuse scheme (drstencil_2d.hpp:180-228): store the  */
                              /* forward sum Dist rows ahead, add the backward sum (csrc/kernels/  */
                              /* drs_reuse.cuh); honours --dist / --merge-forward / --bx/--by/--sn */

typedef struct drs_stencil drs_stencil; /* DRStencil_2d / DRStencil (drstencil_2d.hpp:14-45, drstencil.hpp:14-49) */
typedef struct drs_plan drs_plan;       /* one specialised, compiled sweep == one emitted dr_<name> + its launch shape */

/* The generator's command-line knobs, same names and defaults as main.cpp:12-56.
 * drs_knobs_default() fills the reference defaults; fields after `check` are extensions. */
typedef struct drs_knobs {
    int step;          /* --step            1  */
    int dist;          /* --dist            0 = derive */
    int streaming;     /* --streaming       0  */
    int bx, by;        /* --bx --by         16 16 */
    int sn;            /* --sn              16 */
    int stream_unroll; /* --stream-unroll   4  */
    int block_merge_x, block_merge_y;   /* 1 1 */
    int cyclic_merge_x, cyclic_merge_y; /* 1 1 */
    int prefetch;      /* --prefetch        0  */
    int merge_forward; /* --merge-forward   5  */
    int check;         /* --check           0  */
    /* extensions */
    int dtype;         /* --dtype f64|f32   DRS_F64 */
    int fuse;          /* --fuse temporal|algebraic   DRS_FUSE_TEMPORAL */
    int explicit_mask; /* bit i set: knob i (in the order above, step = bit 0) was given explicitly;
                          knobs not given explicitly are chosen by the engine's B200 heuristics */
    /* engine-only tile overrides (0 = let the engine choose); the tuner's extra axes:
     * [0] ring stages  [1] __launch_bounds__ minimum blocks per SM  [2] warps per CTA
     * [3] rows per thread in 3D  [4] rows per TMA stage in 2D  [5] 128-bit vectors per thread in 2D
     * [6] bit 0: no row factorisation, bit 1: 3D temporal depth as per-sub-step launches instead of the fused kernel,
 *     bits 2-3 / 4-5: warps of a CTA along x / y, minus one, that share one input ring in the
 *     single-step 3D sweep (0 = one private ring per warp) */
    int reserved[7];
} drs_knobs;

/* Geometry the engine chose for a plan (for logs, the tuner and bench.py). */
typedef struct drs_plan_info {
    int dim, dtype, step, fuse;
    long long L, M, N;
    int halo;              /* Halo macro: ring left untouched per sweep                       */
    int npoints;           /* points of the operator one sub-step evaluates                   */
    int timesteps_per_sweep;
    int warps_per_cta, tile_x, tile_y, chunk, stages, rows_per_stage;
    int grid_x, grid_y, grid_z, block;
    int smem_bytes, regs_per_thread, spill_bytes;
    double redundancy;     /* computed points / useful points                                 */
    char kernel_name[96];
} drs_plan_info;

void drs_knobs_default(drs_knobs *k);

/* ---- stencil description: replaces get_stencil / fusing / dataReuse -------------------- */

/* drstencil_2d.hpp:48-73, drstencil.hpp:52-78 */
int drs_stencil_from_file(const char *stc_path, int is3d, drs_stencil **out);
/* same object from memory: offsets = npoints x dim ints, slowest axis first ((j,i) or (k,j,i)) */
int drs_stencil_from_points(int dim, const int *offsets, const double *coefs, int npoints,
                            long long L, long long M, long long N, int iterations, drs_stencil **out);
void drs_stencil_destroy(drs_stencil *s);
/* kernel identifier suffix: dr_<name>, gold_<name>.  From a file it is the file name minus its last
 * four characters (main.cpp:243-244,264-265); from points it defaults to "stencil". */
int drs_stencil_set_name(drs_stencil *s, const char *name);
int drs_stencil_set_size(drs_stencil *s, long long L, long long M, long long N, int iterations);
/* drstencil_2d.hpp:231-251 (fusing) -- composes the base operator `step` times (step >= 1) */
int drs_stencil_compose(drs_stencil *s, int step);
/* sizes: dims[0..2] = L, M, N ; returns iterations through *iterations */
int drs_stencil_size(const drs_stencil *s, long long dims[3], int *iterations);
/* current (composed) operator in evaluation order; offsets written as npoints x 3 (k, j, i);
 * coefs are the doubles denoted by the 6-significant-digit literals the reference would print
 * (drstencil_2d.hpp:174).  Pass NULL buffers to query the count.  Returns npoints or < 0. */
int drs_stencil_terms(const drs_stencil *s, int *offsets3, double *coefs, int capacity);
/* coefficient literal text of term q ("%g"), for emitters and tests */
int drs_stencil_term_text(const drs_stencil *s, int q, char *buf, size_t buflen);
/* drstencil_2d.hpp:82-97,180-228,254-269: Halo, Dist, Range and partition sizes.
 * sizes[0..3] = |forward_slow|, |forward_mid| (3D forward_j), |forward_fast| (forward_i), |backward|.
 * Returns DRS_E_NOREUSE when the reference would stop with "No data to reuse". */
int drs_stencil_analyze(const drs_stencil *s, int dist, int merge_forward, int *halo, int *dist_out,
                        int *range, int sizes[4]);

/* ---- plan: replaces codeGen_2d::output / codeGen::output + nvcc ------------------------- */

/* Specialises and compiles the sm_100a sweep kernel for (stencil, knobs).  The stencil must be
 * un-composed; knobs->step selects the depth.  Needs no GPU until the first sweep. */
int drs_plan_create(const drs_stencil *s, const drs_knobs *k, drs_plan **out);
void drs_plan_destroy(drs_plan *p);
int drs_plan_get_info(const drs_plan *p, drs_plan_info *info);
/* the CUDA C++ translation unit that was specialised (what `drstencil -o` writes, minus main()) */
const char *drs_plan_source(const drs_plan *p);
/* why a requested mode was changed (e.g. temporal -> composed operator), "" if it was not */
const char *drs_plan_note(const drs_plan *p);
/* key of the compiled cubin in the on-disk cache (<cache dir>/<key>.cubin) */
const char *drs_plan_cache_key(const drs_plan *p);
/* the translation unit / cache key of the exact pair kernel drs_run uses on this plan, "" if it uses none */
const char *drs_plan_pair_source(const drs_plan *p);
const char *drs_plan_pair_cache_key(const drs_plan *p);
/* the translation unit / cache key of the slab entry drslab_<name> of a 2D plan, generated and compiled (NVRTC, no GPU
 * needed) by drs_plan_set_slab; "" for every other plan (3D plans carry drslab_ in their main unit) */
const char *drs_plan_slab_source(const drs_plan *p);
const char *drs_plan_slab_cache_key(const drs_plan *p);
/* the translation unit / cache key of the slab pair entry drslabpair_<name>, generated and compiled (NVRTC, no GPU
 * needed) by drs_plan_set_slab_pairs; "" for every other plan */
const char *drs_plan_slab_pair_source(const drs_plan *p);
const char *drs_plan_slab_pair_cache_key(const drs_plan *p);

/* one `dr_<name><<<grid, block>>>(d_in, d_out)` (codegen_2d.hpp:606): advances the interior
 * [Halo, dim-Halo) by `step` timesteps; the Halo ring of d_out is not written.  d_in != d_out.
 * `stream` is a cudaStream_t (NULL = default stream). */
int drs_sweep(drs_plan *p, const void *d_in, void *d_out, void *stream);
/* one `gold_<name><<<...>>>` (codegen_2d.hpp:666-688, codegen.hpp:637-660): the naive
 * one-thread-per-point evaluation of the composed operator, for on-device self-checks */
int drs_gold_sweep(drs_plan *p, const void *d_in, void *d_out, void *stream);
/* the emitted host loop (codegen_2d.hpp:610-613): for (t = 0; t < iterations; t += 2*step)
 * { sweep(A,B); sweep(B,A); } -- result is in A.  Writes the number of sweeps to *sweeps.
 * On 3D step-1 plans whose arrays are >= 1 GiB each (16-byte row pitch, an operator the depth-2 tile fits) the
 * sweeps run as exact pair launches -- one kernel computes two sweeps, bit for bit, with each level's ring taken from
 * the buffer that level lives in -- followed by two or four single sweeps; A and B end exactly as after the plain
 * loop (drs_plan_pair_split).  After drs_plan_set_pairs(p, 1) the same holds for every step-1 plan that has a pair
 * kernel, 2D plans and 3D plans below 1 GiB included.  drs_run on a slab plan (drs_plan_set_slab,
 * drs_plan_set_slab_pairs) never makes pair launches: it is the loop of drs_sweep, boundary planes pushed to the
 * neighbours' ghost planes and no step flags. */
int drs_run(drs_plan *p, void *d_a, void *d_b, int iterations, void *stream, int *sweeps);
/* Opt-in exact pair launches.  enable = 1: drs_run (direct launches and graph replay alike) and the plain
 * copy-sweep-copy drs_run_host (h_b given, or streaming off) run the sweeps as drs_plan_pair_split's pair launches and
 * single sweeps wherever the plan has a pair kernel: on 2D plans the 2D pair unit (kernels/pair2d/drs_pair2d.cuh),
 * generated and compiled here (NVRTC, no GPU needed); on 3D plans the pair unit without its 1 GiB size rule (a no-op
 * where the plan already pairs).  enable = 0 restores the default rule.  drs_plan_pair_source, drs_plan_pair_cache_key
 * and drs_plan_pair_split follow the setting, and so does the streamed drs_run_host (which pairs wherever drs_run
 * does); drs_sweep, drs_gold_run, the slab calls and drs_emit_program do not.  DRS_E_ARG, with the reason, for
 * plans without a pair kernel: step > 1 or per-sub-step launches, `--fuse reuse`, the naive kernel, an unaligned
 * row pitch, an operator whose depth-2 strip or tile keeps no useful columns or whose x extent one lane's shuffle
 * does not reach (2D); and for slab plans, which have drs_plan_set_slab_pairs.  Drops the plan's cached drs_run graphs. */
int drs_plan_set_pairs(drs_plan *p, int enable);
/* how drs_run splits the sweeps of `iterations` timesteps: *pairs pair launches, then *singles single sweeps
 * (*pairs = 0 on plans without pair launches, slab plans included); returns the number of sweeps.  Needs no GPU. */
int drs_plan_pair_split(const drs_plan *p, int iterations, int *pairs, int *singles);
/* drs_run replays its launches as one CUDA graph per (d_a, d_b, sweep count) -- same kernels, same
 * order, without the gap between dependent launches (matters for grids as small as 4096^2).  On
 * by default; a stream that is itself being captured always gets plain launches.  0 switches it off. */
int drs_plan_set_graph(drs_plan *p, int enable);
/* same schedule with the gold kernel (codegen_2d.hpp:638-642) */
int drs_gold_run(drs_plan *p, void *d_a, void *d_b, int iterations, void *stream, int *sweeps);
/* the whole emitted main() data path on HOST buffers (codegen_2d.hpp:572-583,604-619,647):
 * H2D of a and b, the schedule, D2H of a.  h_a/h_b hold L*M*N elements of the plan's dtype;
 * h_b == NULL stands for the all-zero second buffer the reference always uses (common.hpp:34-45)
 * and is cleared on the device instead of being copied.
 * With h_b == NULL the three phases are overlapped by time skewing along the slow axis: the grid
 * is cut into blocks of planes (rows in 2D), each block runs the whole schedule with its output
 * range sliding down one Halo per sweep while later blocks upload and earlier ones download
 * (pinned host memory needed for the overlap; results are bit-identical to the plain sequence).
 * On plans where drs_run makes pair launches the blocks run drs_run's launch sequence -- the pair launches of
 * drs_plan_pair_split, then the single sweeps -- with the range sliding two Halos per pair launch (and two at the
 * first single sweep after them), on blocks at least 4*Halo thick.
 * *device_ms = device time from the first copy to the last, CUDA events. */
int drs_run_host(drs_plan *p, void *h_a, void *h_b, int iterations, float *device_ms);
/* block thickness of the streamed drs_run_host in slow-axis units: 0 = chosen by the engine
 * (>= 32 MiB, about 16 blocks), < 0 = plain copy-sweep-copy, > 0 = as given (raised to 2*Halo, or to 4*Halo when
 * the run makes pair launches) */
int drs_plan_set_host_block(drs_plan *p, long long units);
/* the step list the streamed drs_run_host would execute for `iterations` (needs no GPU): records of five
 * values {kind (0 upload, 1 sweep, 2 download, 3 pair launch), block, launch (1-based index in drs_run's launch
 * sequence; odd: A -> B; on plans without pair launches the sweep number), lo, hi} with [lo, hi) the slow-axis
 * range copied / stored by the launch; per block: its upload, its launches, its download.  Returns the
 * number of records (pass NULL to query), 0 when the plain sequence would run. */
int drs_plan_host_schedule(const drs_plan *p, int iterations, long long *records5, int capacity);
/* The step list one rank of a slab-decomposed host-buffer run executes so that its copies overlap its sweeps
 * like drs_run_host does on one GPU (needs no GPU).  The plan must be a slab (drs_plan_set_slab); up_skew = 0 for
 * even ranks (blocks bottom-up, ranges sliding down), 1 for odd ranks (the mirror image), so that the blocks meeting
 * at a face run in lockstep.  Records of six values {kind, block, sweep, lo, hi, faces}, local plane indices; faces
 * is a bit set: 1 / 2 wait for the lower / upper neighbour's flag >= sweep before the launch, 4 / 8 signal sweep + 1
 * to it afterwards, 16 / 32 (uploads) push the level-0 face planes to it and signal 1.  Returns the number of
 * records (NULL to query), 0 when the plain sequence applies. */
int drs_plan_slab_schedule(const drs_plan *p, int iterations, int up_skew, long long *records6, int capacity);
/* checkError2D / checkError3D (common.hpp:47-102) on device buffers: res[0] = max |a-b| (floored
 * at 1e-13 like the reference), res[1] = RMS, over [Halo, dim-Halo) */
int drs_check_error(drs_plan *p, const void *d_out, const void *d_ref, double res[2]);
/* waits for `stream` and reports DRS_E_KERNEL if a sweep's pipeline watchdog fired (the sweep
 * entry points themselves never synchronise) */
int drs_plan_sync_check(drs_plan *p, void *stream);
/* number of kernels this plan has launched since creation (bench.py's gpu_launches) */
long long drs_plan_launch_count(const drs_plan *p);

/* ---- slab decomposition along the slowest axis (extension; the reference is single-GPU) -- */

/* Declares that this plan's arrays are a slab: planes (3D) / rows (2D) [lo, hi) of a global grid
 * with `global_slow` planes (rows), stored with `ghost` = step*radius extra planes (rows) on each side, i.e.
 * the local array holds (hi - lo + 2*ghost) planes (rows).  The global frozen ring applies only at the
 * global faces.  Must be called before the first sweep.  On a 2D plan with the TMA sweep this generates and
 * compiles the slab unit (drs_plan_slab_source). */
int drs_plan_set_slab(drs_plan *p, long long global_slow, long long lo, long long hi);
/* Like drs_plan_set_slab, for a PAIR slab: the ghost regions are 2*Halo planes deep, i.e. the local array holds
 * (hi - lo + 4*Halo) planes, and drs_run_slab runs the sweeps as exact pair launches (two sweeps per launch, bit for
 * bit) followed by two or four single sweeps (drs_plan_slab_split), each pair launch exchanging one double-depth halo.
 * Every single sweep (drs_sweep, drs_run) pushes 2*Halo planes.  Generates and compiles the slab pair unit
 * (drs_plan_slab_pair_source).  DRS_E_ARG for 2D plans, step > 1 or per-sub-step launches, an unaligned row pitch,
 * `--fuse reuse`, the naive kernel, operators whose depth-2 tile keeps no useful columns, a wrong local size and a
 * plan that is already a slab.  drs_run_host_slab and drs_plan_slab_schedule refuse pair slabs. */
int drs_plan_set_slab_pairs(drs_plan *p, long long global_slow, long long lo, long long hi);
/* how drs_run_slab splits the sweeps of `iterations` timesteps: *pairs pair launches, then *singles single sweeps
 * (*pairs = 0 except on pair slabs); the split depends on the sweep count only, so every rank runs the same launch
 * sequence.  Returns the number of sweeps.  Needs no GPU. */
int drs_plan_slab_split(const drs_plan *p, int iterations, int *pairs, int *singles);
/* One pair launch on a pair slab whose peers are set (the pair counterpart of drs_sweep): the level in d_in advanced
 * by two sweeps on the owned planes of d_out, the 2*Halo boundary planes pushed to the neighbours' deep ghost planes;
 * no step flags.  d_in and d_out are the two arrays given to drs_plan_set_peers; level 0's global ring is taken from
 * the first, level 1's from the second, as in drs_run_slab. */
int drs_sweep_pair(drs_plan *p, const void *d_in, void *d_out, void *stream);
/* Fused halo push: while sweeping into my_bases[b], the kernel stores its boundary planes (3D) / rows (2D) a
 * second time, straight into the neighbours' ghost planes / rows over NVLink.  lower_bases / upper_bases
 * are the *neighbours' array bases* (same ping-pong order, mapped into this process with
 * drs_ipc_import), NULL where there is no neighbour; lower_lo / upper_lo are the neighbours' first
 * owned global planes / rows (their `lo`).  On a 2D plan every sweep then runs the slab entry drslab_<name>; a 2D
 * slab plan without peers keeps the plain kernel and frozen ghost rows.  DRS_E_ARG for plans without a slab kernel:
 * `--fuse reuse` and the naive kernel of operators too deep for the TMA ring. */
int drs_plan_set_peers(drs_plan *p, void *const my_bases[2], void *const lower_bases[2],
                       void *const upper_bases[2], long long lower_lo, long long upper_lo);
/* Cross-GPU step flags.  Each rank owns a device array of two 64-bit slots (slot 0 written by its lower
 * neighbour, slot 1 by its upper neighbour), zero-initialised, allocated with drs_device_malloc and exported with
 * drs_ipc_export.  drs_plan_set_flags hands the plan this rank's array and the two remote slots it writes:
 * lower_flag = the lower neighbour's slot 1, upper_flag = the upper neighbour's slot 0 (NULL where there is no
 * neighbour).  Flag values are monotone over the life of the plan (sweeps run so far), never reset. */
int drs_plan_set_flags(drs_plan *p, const void *my_flags, void *lower_flag, void *upper_flag);
/* This rank's share of the emitted host loop (codegen.hpp:575-589, codegen_2d.hpp:610-613) on a slab-decomposed grid:
 * `for (t = 0; t < iterations; t += 2*step) { sweep(A,B); sweep(B,A); }` over the arrays given to drs_plan_set_peers,
 * ONE kernel launch per sweep, replayed as a CUDA graph.  The sweep kernel does the whole exchange itself: tiles next
 * to a neighbour's slab wait (ld.acquire.sys) until that neighbour's boundary tiles of the previous sweep are done,
 * boundary planes (rows in 2D) are stored a second time into the neighbour's ghost planes over NVLink, and the last boundary
 * tile of a face releases the next flag value (st.release.sys); boundary tiles are scheduled first, so the
 * signal leaves early and the next sweep does not wait.  Every rank must call it with the same `iterations`;
 * after new data was written into the arrays (ghost planes included) the ranks must pass a barrier of the
 * caller's before the next call.  Writes the number of sweeps to *sweeps.  On a pair slab (drs_plan_set_slab_pairs)
 * the sweeps run as drs_plan_slab_split's pair launches and single sweeps, one launch each, and the flag values count
 * launches instead of sweeps. */
int drs_run_slab(drs_plan *p, int iterations, void *stream, int *sweeps);
/* This rank's share of a slab-decomposed HOST-buffer run (the executor of drs_plan_slab_schedule): h_own = the
 * rank's own planes (rows in 2D; pinned for overlap), result written back in place; uploads, sweeps and downloads overlap
 * by time-skewed blocks, the faces run in lockstep with the neighbours through the plan's flags.  The device
 * arrays are the ones given to drs_plan_set_peers (second one zero-initialised by the caller).  Ranks pass a
 * barrier of the caller's between calls.  up_skew as for drs_plan_slab_schedule.  *device_ms as drs_run_host. */
int drs_run_host_slab(drs_plan *p, void *h_own, int iterations, int up_skew, float *device_ms);
/* The protocol's two halves as separate one-thread kernels (what drs_run_slab fuses into the sweep; used by
 * drs_run_host_slab and kept for A/B measurements): drs_signal_peers enqueues, after the work already on
 * `stream`, a system-scope release store of `value` into the given remote slots; drs_wait_flags enqueues a wait
 * until the selected slots of `my_flags` hold >= value. */
int drs_signal_peers(drs_plan *p, void *lower_flag, void *upper_flag, long long value, void *stream);
int drs_wait_flags(drs_plan *p, const void *my_flags, int wait_lower, int wait_upper, long long value, void *stream);
/* CUDA IPC plumbing so that one process per GPU can map a neighbour's buffer.  Buffers to be
 * exported must come from drs_device_malloc (a whole cudaMalloc allocation). */
int drs_device_malloc(size_t bytes, void **d_ptr);
int drs_device_free(void *d_ptr);
int drs_device_upload(void *d_dst, const void *h_src, size_t bytes);   /* blocking cudaMemcpy H2D */
int drs_device_download(void *h_dst, const void *d_src, size_t bytes); /* blocking cudaMemcpy D2H */
int drs_ipc_export(void *d_ptr, unsigned char handle[64]);
int drs_ipc_import(const unsigned char handle[64], void **d_ptr);
int drs_ipc_close(void *d_ptr);

/* ---- emitters: replaces `drstencil -o out.cu` ------------------------------------------- */

/* Writes a standalone CUDA program (kernel specialisation + main() with the reference's stdout
 * lines, codegen_2d.hpp:571,602,617-618,624,650) to `path`. */
int drs_emit_program(const drs_stencil *s, const drs_knobs *k, const char *kernel_name, const char *path);

/* ---- misc -------------------------------------------------------------------------------- */
const char *drs_last_error(void);
const char *drs_version(void);
/* which NVRTC the library compiles its kernels with ("NVRTC 12.8 (<path>)"): one pinned copy for every consumer */
const char *drs_compiler(void);
int drs_device_count(void);
/* makes CUDA device `ordinal` current for the calling thread (one process per GPU: LOCAL_RANK); a plan is bound
 * to the device that is current at its first sweep */
int drs_set_device(int ordinal);
/* pre-compiles without a GPU and stores the cubin in the on-disk cache (build step) */
int drs_plan_warm_cache(const drs_stencil *s, const drs_knobs *k);
void drs_set_cache_dir(const char *dir);

#ifdef __cplusplus
}
#endif
#endif /* DRSTENCIL_H_ */
