// drstencil -- command-line generator of the B200 stencil engine.
//
// Drop-in for the reference CLI (/root/reference/main.cpp:10-280): same option names, defaults,
// positional rule (the .stc file is ALWAYS the last argument) and exit behaviour:
//   no argument                         "Please specify the .stc file."            rc 0   (main.cpp:61-64)
//   --help / -h as first argument       usage                                      rc 0   (main.cpp:65-117)
//   valued option in the last-but-one slot  "Illegal input."                       rc 255 (exit(-1))
//   `-o` in the last-but-one slot       silently ignored                                  (main.cpp:119-122)
//   unknown option                      "Illegal input."                           rc 0   (main.cpp:226-229)
//   unreadable .stc                     "Error opening stencil file."              rc 255 (main.cpp:240-241)
//   no slow-axis forward set            "No data to reuse. You can try another dist." rc 1
//                                                                       (drstencil_2d.hpp:217-220)
//   2*Halo >= bx*mx with forward_i (or, 3D, >= by*my with forward_j)  "Invalid configuration!" rc 255
//                                                                       (codegen_2d.hpp:52-56, codegen.hpp:50-55)
// On success it writes a CUDA program to -o (default out.cu) -- see csrc/capi/emit_program.hpp.
// Extensions (not in the reference): --dtype, --fuse, --run, --pairs, --info, --allow-no-reuse and the
// engine-only tile overrides --stages --warps --min-blocks --vectors --rows-3d --rows-per-stage.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <iostream>
#include <string>
#include <vector>

#include "drstencil.h"


static const char* kHelp = R"(
    Generate a B200 (sm_100a) stencil sweep from a .stc description.

    Usage: drstencil [options] <input_stcfile>
Options (same names and defaults as the reference generator):

-o <file>               Name of the output CUDA file (out.cu by default).
--3d                    3D mode.
--step <num>            Time steps advanced per sweep (1 by default): in-kernel temporal
                        blocking, or the composed operator with --fuse algebraic.
--dist <num>            Reuse distance of the reference's forward/backward partition
                        (reported only: this engine writes each output once).
--streaming             Accepted; the engine always streams along the slowest axis.
--bx <num>  --by <num>  Block shape (16 16): bx*by/32 warps per CTA (--streaming: bx/32).
--sn <num>              Slow-axis outputs per tile (16 in the reference; B200 heuristic if omitted).
--stream-unroll <num>   Rows per TMA stage in 2D (4 by default).
--block-merge-x <num>   128-bit vectors of adjacent columns per thread in 2D (1 or 2).
--block-merge-y <num>   3D: rows per thread = 4 * num.
--cyclic-merge-x <num>  Accepted (no effect).
--cyclic-merge-y <num>  3D: rows per thread = 4 * num.
--prefetch              Deeper TMA ring (8 stages).
--merge-forward <num>   Threshold of the reference's partition merge (5 by default; reported only).
--check                 Emit the gold kernel and the error check.
--gold                  Accepted (no effect, as in the reference).
--help  (-h)            Print this help.

Extensions:
--dtype <f64|f32>       Element type (f64 by default; the reference is fp64 only).
--fuse <temporal|algebraic|reuse>   Meaning of --step (temporal by default); reuse = the reference's
                        forward/backward data-reuse evaluation of the composed operator (A/B mode).
--run                   Do not emit: run the emitted program's host loop on the GPU through
                        libdrstencil.so and print the same lines.
--pairs                 With --run: the host loop runs as exact pair launches (two bit-exact
                        single-step sweeps per launch, drs_plan_set_pairs); an error where the plan
                        has no pair kernel.  No effect on the emitted program.
--info                  Print the chosen tile geometry and the reference macros (Halo Dist Range).
--allow-no-reuse        Do not stop where the reference prints "No data to reuse".
--stages --warps --min-blocks --vectors --rows-3d --rows-per-stage <num>   tile overrides.
--share-x --share-y <1..4>   warps of a CTA along x / y that share one input ring (3D, single step).
        )";

static int illegal_exit() {
    std::cout << "Illegal input." << std::endl;
    exit(-1);
}

int main(int argc, char** argv) {
    if (argc < 2) {
        std::cout << "Please specify the .stc file." << std::endl;
        return 0;
    }
    if (!strcmp(argv[1], "--help") || !strcmp(argv[1], "-h")) {
        std::cout << kHelp << std::endl;
        return 0;
    }
    drs_knobs k;
    drs_knobs_default(&k);
    std::string out_name = "out.cu";
    bool is3d = false, run = false, pairs = false, info = false, allow_no_reuse = false;
    struct Opt { const char* name; int* value; int bit; int reserved; };
    const Opt valued[] = {
        {"--step", &k.step, 0, -1}, {"--dist", &k.dist, 1, -1}, {"--bx", &k.bx, 3, -1}, {"--by", &k.by, 4, -1},
        {"--sn", &k.sn, 5, -1}, {"--stream-unroll", &k.stream_unroll, 6, -1},
        {"--block-merge-x", &k.block_merge_x, 7, -1}, {"--block-merge-y", &k.block_merge_y, 8, -1},
        {"--cyclic-merge-x", &k.cyclic_merge_x, 9, -1}, {"--cyclic-merge-y", &k.cyclic_merge_y, 10, -1},
        {"--merge-forward", &k.merge_forward, 12, -1},
        {"--stages", nullptr, -1, 0}, {"--min-blocks", nullptr, -1, 1}, {"--warps", nullptr, -1, 2},
        {"--rows-3d", nullptr, -1, 3}, {"--rows-per-stage", nullptr, -1, 4}, {"--vectors", nullptr, -1, 5},
    };
    for (int i = 1; i < argc - 1; i++) {
        const std::string a = argv[i];
        bool done = false;
        if (a == "-o") { if (i != argc - 2) out_name = argv[++i]; continue; }
        if (a == "--3d") { is3d = true; continue; }
        if (a == "--streaming") { k.streaming = 1; k.explicit_mask |= 1 << 2; continue; }
        if (a == "--prefetch") { k.prefetch = 1; k.explicit_mask |= 1 << 11; continue; }
        if (a == "--check") { k.check = 1; k.explicit_mask |= 1 << 13; continue; }
        if (a == "--gold") continue;
        if (a == "--run") { run = true; continue; }
        if (a == "--pairs") { pairs = true; continue; }
        if (a == "--info") { info = true; continue; }
        if (a == "--allow-no-reuse") { allow_no_reuse = true; continue; }
        if (a == "--share-x" || a == "--share-y") {      // CTA-shared ring (drstencil.h, reserved[6])
            if (i == argc - 2) illegal_exit();
            const int v = atoi(argv[++i]);
            if (v < 1 || v > 4) illegal_exit();
            const int shift = a == "--share-x" ? 2 : 4;
            k.reserved[6] = (k.reserved[6] & ~(3 << shift)) | ((v - 1) << shift);
            continue;
        }
        if (a == "--dtype" || a == "--fuse") {
            if (i == argc - 2) illegal_exit();
            const std::string v = argv[++i];
            if (a == "--dtype") {
                if (v == "f64" || v == "fp64" || v == "double") k.dtype = DRS_F64;
                else if (v == "f32" || v == "fp32" || v == "float") k.dtype = DRS_F32;
                else illegal_exit();
                k.explicit_mask |= 1 << 14;
            } else {
                if (v == "temporal") k.fuse = DRS_FUSE_TEMPORAL;
                else if (v == "algebraic") k.fuse = DRS_FUSE_ALGEBRAIC;
                else if (v == "reuse") k.fuse = DRS_FUSE_REUSE;
                else illegal_exit();
                k.explicit_mask |= 1 << 15;
            }
            continue;
        }
        for (const Opt& o : valued) {
            if (a == o.name) {
                if (i == argc - 2) illegal_exit();
                const int v = atoi(argv[++i]);
                if (o.value) { *o.value = v; k.explicit_mask |= 1 << o.bit; }
                else k.reserved[o.reserved] = v;
                done = true;
                break;
            }
        }
        if (done) continue;
        std::cout << "Illegal input." << std::endl;
        return 0;
    }

    const char* stcfile = argv[argc - 1];
    drs_stencil* st = nullptr;
    if (drs_stencil_from_file(stcfile, is3d ? 1 : 0, &st) != DRS_OK) {
        std::cout << drs_last_error() << std::endl;   // "Error opening stencil file."
        exit(-1);
    }
    // the reference's analysis on the composed operator: Halo / Dist / Range, partition, validity
    drs_stencil* comp = nullptr;
    drs_stencil_from_file(stcfile, is3d ? 1 : 0, &comp);
    if (k.step < 1) k.step = 1;
    drs_stencil_compose(comp, k.step);
    int halo = 0, dist = 0, range = 0, sizes[4] = {0, 0, 0, 0};
    const int arc = drs_stencil_analyze(comp, k.dist, k.merge_forward, &halo, &dist, &range, sizes);
    if (arc == DRS_E_NOREUSE && !allow_no_reuse) {
        std::cout << "No data to reuse. You can try another dist.\n";
        return 1;
    }
    const int mx = k.block_merge_x > k.cyclic_merge_x ? k.block_merge_x : k.cyclic_merge_x;
    const int my = k.block_merge_y > k.cyclic_merge_y ? k.block_merge_y : k.cyclic_merge_y;
    if (arc == DRS_OK) {
        const bool fwd_i = sizes[2] > 0, fwd_j = sizes[1] > 0;
        if ((2 * halo >= k.bx * mx && fwd_i) || (is3d && 2 * halo >= k.by * my && fwd_j)) {
            std::cout << "Invalid configuration!" << std::endl;
            exit(-1);
        }
    }
    if (info) {
        drs_plan* p = nullptr;
        if (drs_plan_create(st, &k, &p) != DRS_OK) { std::cout << drs_last_error() << std::endl; exit(-1); }
        drs_plan_info pi;
        drs_plan_get_info(p, &pi);
        printf("Halo %d Dist %d Range %d  forward_slow %d forward_mid %d forward_fast %d backward %d\n", halo, dist,
               range, sizes[0], sizes[1], sizes[2], sizes[3]);
        printf("kernel %s  points/sub-step %d  timesteps/sweep %d  warps/CTA %d  tile %dx%d  chunk %d  stages %d x %d rows\n",
               pi.kernel_name, pi.npoints, pi.timesteps_per_sweep, pi.warps_per_cta, pi.tile_x, pi.tile_y, pi.chunk,
               pi.stages, pi.rows_per_stage);
        printf("grid %d x %d threads  smem %d B  redundancy %.3f\n", pi.grid_x, pi.block, pi.smem_bytes, pi.redundancy);
        drs_plan_destroy(p);
    }
    if (run) {
        // the emitted main(), executed here: rand()/(RAND_MAX-1) input, 10 warm-up launches, timed loop
        long long dims[3]; int iterations = 0;
        drs_stencil_size(st, dims, &iterations);
        drs_plan* p = nullptr;
        if (drs_plan_create(st, &k, &p) != DRS_OK) { std::cout << drs_last_error() << std::endl; exit(-1); }
        if (pairs && drs_plan_set_pairs(p, 1) != DRS_OK) { std::cout << drs_last_error() << std::endl; exit(-1); }
        puts("Initiating ...");
        const size_t count = (size_t)dims[0] * dims[1] * dims[2];
        const size_t es = k.dtype == DRS_F64 ? 8 : 4;
        void* h_a = malloc(count * es);
        void* h_b = calloc(count, es);
        for (size_t x = 0; x < count; ++x) {
            const double v = (double)rand() / (double)(RAND_MAX - 1);
            if (k.dtype == DRS_F64) ((double*)h_a)[x] = v; else ((float*)h_a)[x] = (float)v;
        }
        auto die = [&]() { printf("CUDA error : %s\n", drs_last_error()); exit(-1); };
        void *in = nullptr, *out = nullptr;
        if (drs_device_malloc(count * es, &in) != DRS_OK || drs_device_malloc(count * es, &out) != DRS_OK) die();
        if (drs_device_upload(in, h_a, count * es) != DRS_OK || drs_device_upload(out, h_b, count * es) != DRS_OK) die();
        puts("GPU computing ...");
        for (int i = 0; i < 10; i++)                       // warm up (idempotent on `out`)
            if (drs_sweep(p, in, out, nullptr) != DRS_OK) die();
        if (drs_plan_sync_check(p, nullptr) != DRS_OK) die();
        struct timespec t0, t1;
        clock_gettime(CLOCK_MONOTONIC, &t0);
        if (drs_run(p, in, out, iterations, nullptr, nullptr) != DRS_OK) die();
        if (drs_plan_sync_check(p, nullptr) != DRS_OK) die();
        clock_gettime(CLOCK_MONOTONIC, &t1);
        puts("GPU finished computing.");
        printf("GPU computation time: %f ms\n", (t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6);
        if (k.check) {
            puts("Checking error ...");
            void *g_in = nullptr, *g_out = nullptr;
            if (drs_device_malloc(count * es, &g_in) != DRS_OK || drs_device_malloc(count * es, &g_out) != DRS_OK) die();
            if (drs_device_upload(g_in, h_a, count * es) != DRS_OK || drs_device_upload(g_out, h_b, count * es) != DRS_OK) die();
            if (drs_gold_run(p, g_in, g_out, iterations, nullptr, nullptr) != DRS_OK) die();
            // checkError2D / checkError3D (common.hpp:47-102) on the host, like the emitted program: running maximum
            // from 1e-13 with the reference's "differ" lines, the index of the maximum, RMS over the interior
            if (drs_device_download(h_a, in, count * es) != DRS_OK || drs_device_download(h_b, g_in, count * es) != DRS_OK) die();
            drs_plan_info pi;
            drs_plan_get_info(p, &pi);
            const long long H = pi.halo, L = dims[0], M = dims[1], N = dims[2];
            const long long k0 = is3d ? H : 0, k1 = is3d ? L - H : 1;
            double error = 0.0, max_error = 1e-13;
            long long mk = 0, mj = 0, mi = 0;
            for (long long kk = k0; kk < k1; kk++)
                for (long long j = H; j < M - H; j++)
                    for (long long i = H; i < N - H; i++) {
                        const size_t x = (size_t)((kk * M + j) * N + i);
                        const double o = k.dtype == DRS_F64 ? ((double*)h_a)[x] : (double)((float*)h_a)[x];
                        const double r = k.dtype == DRS_F64 ? ((double*)h_b)[x] : (double)((float*)h_b)[x];
                        double d = o - r;
                        d = d < 0.0 ? -d : d;
                        error += d * d;
                        if (d > max_error) {
                            if (is3d) printf("Values at index (%lld,%lld,%lld) differ : %.6f and %.6f\n", kk, j, i, r, o);
                            else printf("Values at index (%lld,%lld) differ : %.6f and %.6f\n", j, i, r, o);
                            max_error = d; mk = kk; mj = j; mi = i;
                        }
                    }
            if (is3d) printf("[Test] Max Error : %e @ (%lld,%lld,%lld)\n", max_error, mk, mj, mi);
            else printf("[Test] Max Error : %e @ (,%lld,%lld)\n", max_error, mj, mi);
            const double cnt = (double)(k1 - k0) * (double)(M - 2 * H) * (double)(N - 2 * H);
            printf("[Test] RMS Error: %e\n", sqrt(error / (cnt > 0 ? cnt : 1)));
            drs_device_free(g_in); drs_device_free(g_out);
        }
        drs_device_free(in); drs_device_free(out);
        free(h_a); free(h_b);
        drs_plan_destroy(p);
    } else {
        if (drs_emit_program(st, &k, nullptr, out_name.c_str()) != DRS_OK) {
            std::cout << drs_last_error() << std::endl;
            exit(-1);
        }
    }
    drs_stencil_destroy(comp);
    drs_stencil_destroy(st);
    return 0;
}
