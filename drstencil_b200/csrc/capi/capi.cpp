// libdrstencil.so -- C ABI launch layer of the B200 stencil engine (see include/drstencil.h).
//
// plan creation  : choose_spec -> generate_tu -> NVRTC (sm_100a cubin, cached on disk)
// first sweep    : cubin -> cuModuleLoadData, cuTensorMapEncodeTiled per buffer
// every sweep    : one cuLaunchKernel of dr_<name>
// There is no CPU path: without a CUDA device every compute entry point returns DRS_E_NOGPU.
#include <cuda.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <functional>
#include <map>
#include <mutex>
#include <sstream>
#include <string>
#include <tuple>
#include <vector>

#include "../../../include/drstencil.h"
#include "../core/generate.hpp"
#include "../core/host_schedule.hpp"
#include "../core/stencil.hpp"
#include "emit_program.hpp"

extern const char* const drs_embedded_header_names[];
extern const char* const drs_embedded_header_texts[];
extern const int drs_embedded_header_count;
extern const char* const drs_pair_header_names[];
extern const char* const drs_pair_header_texts[];
extern const int drs_pair_header_count;
extern const char* const drs_slab2d_header_names[];
extern const char* const drs_slab2d_header_texts[];
extern const int drs_slab2d_header_count;
extern const char* const drs_slabpair_header_names[];
extern const char* const drs_slabpair_header_texts[];
extern const int drs_slabpair_header_count;
extern const char* const drs_pair2d_header_names[];
extern const char* const drs_pair2d_header_texts[];
extern const int drs_pair2d_header_count;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) { g_err = msg; return code; }

// ---------------------------------------------------------------------------------------------
// CUDA driver entry points, fetched through the (statically linked) runtime so that the library
// loads on machines without libcuda.so.1
// ---------------------------------------------------------------------------------------------
struct Driver {
    bool ok = false;
    std::string why;
    CUresult (*ModuleLoadData)(CUmodule*, const void*) = nullptr;
    CUresult (*ModuleUnload)(CUmodule) = nullptr;
    CUresult (*ModuleGetFunction)(CUfunction*, CUmodule, const char*) = nullptr;
    CUresult (*FuncSetAttribute)(CUfunction, CUfunction_attribute, int) = nullptr;
    CUresult (*FuncGetAttribute)(int*, CUfunction_attribute, CUfunction) = nullptr;
    CUresult (*LaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned,
                             CUstream, void**, void**) = nullptr;
    CUresult (*TensorMapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill) = nullptr;
    CUresult (*GetErrorString)(CUresult, const char**) = nullptr;
    CUresult (*StreamWriteValue64)(CUstream, CUdeviceptr, cuuint64_t, unsigned int) = nullptr;   // optional
    CUresult (*OccupancyMaxActiveBlocks)(int*, CUfunction, int, size_t) = nullptr;                 // optional (DRS_DEBUG_OCC)
};

Driver& driver() {
    static Driver d;
    static std::once_flag once;
    std::call_once(once, [] {
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess || n == 0) {
            d.why = std::string("no CUDA device: ") + cudaGetErrorString(e);
            cudaGetLastError();
            return;
        }
        cudaFree(0);  // primary context
        auto get = [&](const char* name, void** fp) {
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint(name, fp, cudaEnableDefault, &q) != cudaSuccess || *fp == nullptr) {
                d.why += std::string("driver entry point missing: ") + name + "; ";
                return false;
            }
            return true;
        };
        bool ok = true;
        ok &= get("cuModuleLoadData", (void**)&d.ModuleLoadData);
        ok &= get("cuModuleUnload", (void**)&d.ModuleUnload);
        ok &= get("cuModuleGetFunction", (void**)&d.ModuleGetFunction);
        ok &= get("cuFuncSetAttribute", (void**)&d.FuncSetAttribute);
        ok &= get("cuFuncGetAttribute", (void**)&d.FuncGetAttribute);
        ok &= get("cuLaunchKernel", (void**)&d.LaunchKernel);
        ok &= get("cuTensorMapEncodeTiled", (void**)&d.TensorMapEncodeTiled);
        ok &= get("cuGetErrorString", (void**)&d.GetErrorString);
        {
            cudaDriverEntryPointQueryResult q;
            void* fp = nullptr;
            if (cudaGetDriverEntryPoint("cuStreamWriteValue64", &fp, cudaEnableDefault, &q) == cudaSuccess && fp)
                d.StreamWriteValue64 = (decltype(d.StreamWriteValue64))fp;
            else cudaGetLastError();
            fp = nullptr;
            if (cudaGetDriverEntryPoint("cuOccupancyMaxActiveBlocksPerMultiprocessor", &fp, cudaEnableDefault, &q) == cudaSuccess && fp)
                d.OccupancyMaxActiveBlocks = (decltype(d.OccupancyMaxActiveBlocks))fp;
            else cudaGetLastError();
        }
        d.ok = ok;
    });
    return d;
}

std::string cu_err(CUresult r) {
    const char* s = nullptr;
    if (driver().GetErrorString) driver().GetErrorString(r, &s);
    return s ? s : "unknown CUDA driver error";
}

// ---------------------------------------------------------------------------------------------
// NVRTC, loaded on demand
// ---------------------------------------------------------------------------------------------
struct Nvrtc {
    bool ok = false;
    std::string why, path;
    void* h = nullptr;
    typedef struct _nvrtcProgram* Prog;
    int (*CreateProgram)(Prog*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*CompileProgram)(Prog, int, const char* const*) = nullptr;
    int (*GetCUBINSize)(Prog, size_t*) = nullptr;
    int (*GetCUBIN)(Prog, char*) = nullptr;
    int (*GetProgramLogSize)(Prog, size_t*) = nullptr;
    int (*GetProgramLog)(Prog, char*) = nullptr;
    int (*DestroyProgram)(Prog*) = nullptr;
    int (*Version)(int*, int*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};

Nvrtc& nvrtc() {
    static Nvrtc n;
    static std::once_flag once;
    std::call_once(once, [] {
        // ONE compiler for every consumer of the library (Python, the C++ CLI, C hosts): the copy pinned at build
        // time (DRS_NVRTC_PINNED, an absolute path: _build.py picks the one every measurement of this repo was
        // taken with), not whatever "libnvrtc.so.12" happens to resolve to in the process -- that depended on
        // whether torch had been imported first, and the two copies in this image (12.8 / 12.9) do not produce the
        // same cubins.  DRS_NVRTC=<path> overrides; the bare names are the fallback for other installations.
        std::vector<std::string> names;
        if (const char* e = getenv("DRS_NVRTC")) names.push_back(e);
#ifdef DRS_NVRTC_PINNED
        names.push_back(DRS_NVRTC_PINNED);
#endif
        for (const char* nm : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"})
            names.push_back(nm);
        for (const std::string& nm : names) {
            n.h = dlopen(nm.c_str(), RTLD_NOW | RTLD_LOCAL);
            if (n.h) { n.path = nm; break; }
        }
        if (!n.h) { n.why = "libnvrtc.so.12 not found"; return; }
        auto get = [&](const char* name) { return dlsym(n.h, name); };
        n.CreateProgram = (decltype(n.CreateProgram))get("nvrtcCreateProgram");
        n.CompileProgram = (decltype(n.CompileProgram))get("nvrtcCompileProgram");
        n.GetCUBINSize = (decltype(n.GetCUBINSize))get("nvrtcGetCUBINSize");
        n.GetCUBIN = (decltype(n.GetCUBIN))get("nvrtcGetCUBIN");
        n.GetProgramLogSize = (decltype(n.GetProgramLogSize))get("nvrtcGetProgramLogSize");
        n.GetProgramLog = (decltype(n.GetProgramLog))get("nvrtcGetProgramLog");
        n.DestroyProgram = (decltype(n.DestroyProgram))get("nvrtcDestroyProgram");
        n.Version = (decltype(n.Version))get("nvrtcVersion");
        n.GetErrorString = (decltype(n.GetErrorString))get("nvrtcGetErrorString");
        n.ok = n.CreateProgram && n.CompileProgram && n.GetCUBINSize && n.GetCUBIN && n.GetProgramLogSize &&
               n.GetProgramLog && n.DestroyProgram && n.Version;
        if (!n.ok) n.why = "libnvrtc is missing entry points";
    });
    return n;
}

std::string g_cache_dir;
std::string cache_dir() {
    if (!g_cache_dir.empty()) return g_cache_dir;
    if (const char* e = getenv("DRS_CACHE_DIR")) return e;
    Dl_info info;
    if (dladdr((void*)&cache_dir, &info) && info.dli_fname) {
        std::string p = info.dli_fname;
        size_t s = p.rfind('/');
        return (s == std::string::npos ? std::string(".") : p.substr(0, s)) + "/_jitcache";
    }
    return "/tmp/drs_jitcache";
}

const char* kNvrtcOpts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "--fmad=false",
                            "-default-device", "--ptxas-options=-v"};

// Which unit compile_cubin builds: the plan's main unit, the exact pair kernel's (kernels/pair/ headers), the 2D slab
// entry's (kernels/slab2d/ headers), the slab entry of the pair kernel (kernels/slabpair/ headers) or the 2D pair
// kernel's (kernels/pair2d/ headers).
enum class Unit { MAIN, PAIR, SLAB2D, SLABPAIR, PAIR2D };

// source -> cubin, through the on-disk cache.  The key covers the source, every header the unit may include and the
// options.  The pair and slab units may include their own subdirectory's headers as well; those are part of their
// keys only: the keys of every other unit do not depend on them.
int compile_cubin(const std::string& src, std::vector<char>& cubin, std::string& key_out, Unit unit = Unit::MAIN) {
    std::vector<const char*> names(drs_embedded_header_names, drs_embedded_header_names + drs_embedded_header_count);
    std::vector<const char*> texts(drs_embedded_header_texts, drs_embedded_header_texts + drs_embedded_header_count);
    if (unit == Unit::PAIR) {
        names.insert(names.end(), drs_pair_header_names, drs_pair_header_names + drs_pair_header_count);
        texts.insert(texts.end(), drs_pair_header_texts, drs_pair_header_texts + drs_pair_header_count);
    } else if (unit == Unit::SLAB2D) {
        names.insert(names.end(), drs_slab2d_header_names, drs_slab2d_header_names + drs_slab2d_header_count);
        texts.insert(texts.end(), drs_slab2d_header_texts, drs_slab2d_header_texts + drs_slab2d_header_count);
    } else if (unit == Unit::SLABPAIR) {
        names.insert(names.end(), drs_slabpair_header_names, drs_slabpair_header_names + drs_slabpair_header_count);
        texts.insert(texts.end(), drs_slabpair_header_texts, drs_slabpair_header_texts + drs_slabpair_header_count);
    } else if (unit == Unit::PAIR2D) {
        names.insert(names.end(), drs_pair2d_header_names, drs_pair2d_header_names + drs_pair2d_header_count);
        texts.insert(texts.end(), drs_pair2d_header_texts, drs_pair2d_header_texts + drs_pair2d_header_count);
    }
    std::string all = src;
    for (const char* t : texts) all += t;
    for (const char* o : kNvrtcOpts) all += o;
    int maj = 0, min = 0;
    Nvrtc& n = nvrtc();
    if (n.ok) n.Version(&maj, &min);
    char key[64];
    std::snprintf(key, sizeof key, "%016llx_%d_%d", (unsigned long long)drs::fnv1a(all), maj, min);
    key_out = key;
    const std::string dir = cache_dir();
    const std::string path = dir + "/" + key + ".cubin";
    {
        std::ifstream f(path, std::ios::binary);
        if (f) {
            cubin.assign(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
            if (!cubin.empty()) return DRS_OK;
        }
    }
    if (!n.ok) return fail(DRS_E_COMPILE, "NVRTC unavailable: " + n.why);
    Nvrtc::Prog prog = nullptr;
    int r = n.CreateProgram(&prog, src.c_str(), "drs_generated.cu", (int)names.size(), texts.data(), names.data());
    if (r != 0) return fail(DRS_E_COMPILE, "nvrtcCreateProgram failed");
    r = n.CompileProgram(prog, (int)(sizeof kNvrtcOpts / sizeof kNvrtcOpts[0]), kNvrtcOpts);
    size_t logn = 0;
    n.GetProgramLogSize(prog, &logn);
    std::string log(logn, '\0');
    if (logn > 1) n.GetProgramLog(prog, &log[0]);
    if (r != 0) {
        n.DestroyProgram(&prog);
        return fail(DRS_E_COMPILE, std::string("NVRTC: ") + (n.GetErrorString ? n.GetErrorString(r) : "error") + "\n" + log);
    }
    size_t sz = 0;
    n.GetCUBINSize(prog, &sz);
    cubin.resize(sz);
    n.GetCUBIN(prog, cubin.data());
    n.DestroyProgram(&prog);
    mkdir(dir.c_str(), 0755);
    {
        std::ofstream lf(dir + "/" + key + ".log");
        lf << log.c_str();
    }
    const std::string tmp = path + ".tmp" + std::to_string((long)getpid());
    {
        std::ofstream f(tmp, std::ios::binary);
        f.write(cubin.data(), (std::streamsize)cubin.size());
    }
    rename(tmp.c_str(), path.c_str());
    return DRS_OK;
}

// Params as the kernels see it (drs_common.cuh: struct Params) -- keep the two in step.
struct DevParams {
    const void* in;
    void* out;
    long long L, M, N;
    long long slow_lo, slow_hi;
    int halo;
    int nxs, nys, nzs;
    int chunk;
    int* fault;
    void* peer_lo;
    void* peer_hi;
    long long push_lo0, push_lo1, peer_lo_shift;
    long long push_hi0, push_hi1, peer_hi_shift;
    // in-kernel slab protocol (drs_run_slab)
    const long long* my_flags;
    long long* lower_flag;
    long long* upper_flag;
    const long long* seq_base;
    unsigned int* face_cnt;
    long long face_lo_end, face_hi_begin;
    int seq_off;
    int face_lo_chunks, face_hi_chunks;
    unsigned int face_lo_units, face_hi_units;
};

}  // namespace

struct drs_stencil {
    drs::Stencil st;
    std::string name = "stencil";
};

struct drs_plan {
    drs::Stencil st;         // base stencil + sizes
    drs_knobs knobs;
    drs::KernelSpec spec;
    std::string source, cache_key;
    std::vector<char> cubin;
    // exact pair launches of drs_run (generate.hpp: pair_spec, and pair_spec2d after drs_plan_set_pairs): their own
    // unit, cubin, module and tensor maps.  Every pair module loaded stays loaded, by cache key, until the plan is
    // destroyed: drs_plan_set_pairs may switch units while launches from the previous one are still queued.
    bool pair = false;
    drs::KernelSpec pspec;
    std::string pair_source, pair_key;
    std::vector<char> pair_cubin;
    std::map<std::string, std::pair<CUmodule, CUfunction>> pmods;
    CUfunction f_pair = nullptr;
    std::map<const void*, CUtensorMap> ptmaps;
    // 2D slab plans (generate.hpp: has_slab2d_unit): the unit of drslab_, generated and compiled by drs_plan_set_slab, its
    // module loaded with the plan's device state.  The tensor maps are the main kernel's.
    std::string slab_source, slab_key;
    std::vector<char> slab_cubin;
    CUmodule smod = nullptr;
    // pair slabs (drs_plan_set_slab_pairs): ghost regions of 2 * Halo planes, and drs_run_slab runs pair launches of
    // drslabpair_ (geometry pspec, tensor maps ptmaps); its unit is compiled by drs_plan_set_slab_pairs, its module
    // loaded with the plan's device state
    bool slab_pairs = false;
    std::string slabpair_source, slabpair_key;
    std::vector<char> slabpair_cubin;
    CUmodule spmod = nullptr;
    CUfunction f_slabpair = nullptr;
    // device state (bound at first use)
    bool loaded = false;
    int device = -1;
    CUmodule mod = nullptr;
    // f_slab: drslab_, from the main module (3D) or from smod (2D)
    CUfunction f_sweep = nullptr, f_slab = nullptr, f_gold = nullptr, f_check = nullptr, f_signal = nullptr, f_wait = nullptr;
    int regs = 0, spill = 0;
    int* d_fault = nullptr;
    double* d_res = nullptr;
    std::map<const void*, CUtensorMap> tmaps;
    void* h_dev[2] = {nullptr, nullptr};  // buffers owned by drs_run_host
    bool h_dev_b_ring_zero = false;       // h_dev[1]'s frozen ring still holds the zeros it was cleared to
    long long host_block = 0;             // drs_plan_set_host_block: 0 = auto, < 0 = no streaming
    cudaStream_t hs_up = nullptr, hs_run = nullptr, hs_dn = nullptr;   // streams of the streamed host runs
    void* scratch[2] = {nullptr, nullptr};  // intermediate time levels of multi-launch 3D temporal sweeps
    long long launches = 0;
    // drs_run and drs_run_slab replay their launch sequences as CUDA graphs (run_graph), one per A, B, sweep
    // count and sequence (true: drs_run_slab's; a slab plan may run either on the same buffers)
    bool use_graph = true;
    cudaStream_t cap_stream = nullptr;
    struct RunGraph { cudaGraphExec_t exec; int kernels; };
    std::map<std::tuple<const void*, const void*, int, bool>, RunGraph> graphs;
    // slab mode
    bool slab = false;
    long long g_slow = 0, lo = 0, hi = 0;
    void* my_bases[2] = {nullptr, nullptr};
    void* lower_bases[2] = {nullptr, nullptr};
    void* upper_bases[2] = {nullptr, nullptr};
    long long lower_lo = 0, upper_lo = 0;
    // in-kernel step flags of drs_run_slab (drs_plan_set_flags): caller-owned flag words, plan-owned
    // sequence base + face counters; slab_seq = sweeps run so far (flag values are monotone)
    const void* my_flags = nullptr;
    void* lower_flag = nullptr;
    void* upper_flag = nullptr;
    void* d_sync = nullptr;               // { long long seq_base; unsigned face_cnt[2]; }
    long long slab_seq = 0;

    long long local_slow() const { return spec.dim == 3 ? st.L : st.M; }
    long long ghost() const { return slab_pairs ? 2LL * spec.halo : spec.halo; }   // ghost planes per side of a slab
};

namespace {

// The slab pair unit's module and drslabpair_ (once the plan is loaded and has a compiled slab pair unit)
int load_slabpair(drs_plan* p) {
    if (p->slabpair_cubin.empty() || p->spmod) return DRS_OK;
    Driver& d = driver();
    CUresult r = d.ModuleLoadData(&p->spmod, p->slabpair_cubin.data());
    if (r != CUDA_SUCCESS) { p->spmod = nullptr; return fail(DRS_E_CUDA, "cuModuleLoadData(slab pair): " + cu_err(r)); }
    r = d.ModuleGetFunction(&p->f_slabpair, p->spmod, ("drslabpair_" + p->spec.name).c_str());
    if (r == CUDA_SUCCESS) r = d.FuncSetAttribute(p->f_slabpair, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, p->pspec.smem_bytes());
    if (r != CUDA_SUCCESS) {
        d.ModuleUnload(p->spmod);
        p->spmod = nullptr;
        p->f_slabpair = nullptr;
        return fail(DRS_E_CUDA, "cuModuleGetFunction(drslabpair_): " + cu_err(r));
    }
    return DRS_OK;
}

// The 2D slab unit's module and drslab_, with f_sweep's dynamic shared memory and carve-out (once the plan is loaded and
// has a compiled slab unit; drs_plan_set_slab may come after the first use of the plan)
int load_slab2d(drs_plan* p) {
    const int rc = load_slabpair(p);
    if (rc != DRS_OK) return rc;
    if (p->slab_cubin.empty() || p->smod) return DRS_OK;
    Driver& d = driver();
    CUresult r = d.ModuleLoadData(&p->smod, p->slab_cubin.data());
    if (r != CUDA_SUCCESS) { p->smod = nullptr; return fail(DRS_E_CUDA, "cuModuleLoadData(slab): " + cu_err(r)); }
    r = d.ModuleGetFunction(&p->f_slab, p->smod, ("drslab_" + p->spec.name).c_str());
    if (r == CUDA_SUCCESS) r = d.FuncSetAttribute(p->f_slab, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, p->spec.smem_bytes());
    if (r != CUDA_SUCCESS) {
        d.ModuleUnload(p->smod);
        p->smod = nullptr;
        p->f_slab = nullptr;
        return fail(DRS_E_CUDA, "cuModuleGetFunction(drslab_): " + cu_err(r));
    }
    if (const char* co = std::getenv("DRS_CARVEOUT")) d.FuncSetAttribute(p->f_slab, CU_FUNC_ATTRIBUTE_PREFERRED_SHARED_MEMORY_CARVEOUT, std::atoi(co));
    return DRS_OK;
}

// The current pair unit's module and drpair_ (once the plan is loaded), from pmods when it was loaded before
int load_pair(drs_plan* p) {
    if (!p->pair) { p->f_pair = nullptr; return DRS_OK; }
    auto it = p->pmods.find(p->pair_key);
    if (it == p->pmods.end()) {
        Driver& d = driver();
        CUmodule m = nullptr;
        CUfunction f = nullptr;
        CUresult r = d.ModuleLoadData(&m, p->pair_cubin.data());
        if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuModuleLoadData(pair): " + cu_err(r));
        r = d.ModuleGetFunction(&f, m, ("drpair_" + p->spec.name).c_str());
        if (r == CUDA_SUCCESS) r = d.FuncSetAttribute(f, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, p->pspec.smem_bytes());
        if (r != CUDA_SUCCESS) {
            d.ModuleUnload(m);
            return fail(DRS_E_CUDA, "cuModuleGetFunction(drpair_): " + cu_err(r));
        }
        it = p->pmods.emplace(p->pair_key, std::make_pair(m, f)).first;
    }
    p->f_pair = it->second.second;
    return DRS_OK;
}

int ensure_loaded(drs_plan* p) {
    if (p->loaded) {
        // the module, tensor maps and scratch memory belong to the device that was current at first use
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess || cur != p->device)
            return fail(DRS_E_ARG, "plan is bound to CUDA device " + std::to_string(p->device) + " but device " +
                                       std::to_string(cur) + " is current");
        return load_slab2d(p);
    }
    Driver& d = driver();
    if (!d.ok) return fail(DRS_E_NOGPU, "drstencil needs a CUDA device (no CPU fallback): " + d.why);
    cudaGetDevice(&p->device);
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, p->device);
    if (prop.major != 10) {
        return fail(DRS_E_NOGPU, std::string("kernels are built for sm_100a only; device is ") + prop.name + " (sm_" +
                                     std::to_string(prop.major) + std::to_string(prop.minor) + ")");
    }
    CUresult r = d.ModuleLoadData(&p->mod, p->cubin.data());
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuModuleLoadData: " + cu_err(r));
    const std::string nm = p->spec.name;
    if (p->spec.reuse) {
        r = d.ModuleGetFunction(&p->f_sweep, p->mod, ("dr_" + nm).c_str());
        if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuModuleGetFunction(dr_): " + cu_err(r));
        d.FuncGetAttribute(&p->regs, CU_FUNC_ATTRIBUTE_NUM_REGS, p->f_sweep);
        d.FuncGetAttribute(&p->spill, CU_FUNC_ATTRIBUTE_LOCAL_SIZE_BYTES, p->f_sweep);
    } else if (p->spec.tma_ok) {
        r = d.ModuleGetFunction(&p->f_sweep, p->mod, ("dr_" + nm).c_str());
        if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuModuleGetFunction(dr_): " + cu_err(r));
        const int smem = p->spec.smem_bytes();
        r = d.FuncSetAttribute(p->f_sweep, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, smem);
        if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuFuncSetAttribute(smem): " + cu_err(r));
        if (p->spec.dim == 3) {     // the entry point with the in-kernel slab protocol (drs_run_slab)
            r = d.ModuleGetFunction(&p->f_slab, p->mod, ("drslab_" + nm).c_str());
            if (r == CUDA_SUCCESS) r = d.FuncSetAttribute(p->f_slab, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, smem);
            if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuModuleGetFunction(drslab_): " + cu_err(r));
        }
        d.FuncGetAttribute(&p->regs, CU_FUNC_ATTRIBUTE_NUM_REGS, p->f_sweep);
        d.FuncGetAttribute(&p->spill, CU_FUNC_ATTRIBUTE_LOCAL_SIZE_BYTES, p->f_sweep);
        // development aid: DRS_CARVEOUT=<percent> states a shared-memory carve-out preference for the sweep kernels
        // (default: the driver's own choice)
        if (const char* co = std::getenv("DRS_CARVEOUT")) {
            const int pct = std::atoi(co);
            d.FuncSetAttribute(p->f_sweep, CU_FUNC_ATTRIBUTE_PREFERRED_SHARED_MEMORY_CARVEOUT, pct);
            if (p->f_slab) d.FuncSetAttribute(p->f_slab, CU_FUNC_ATTRIBUTE_PREFERRED_SHARED_MEMORY_CARVEOUT, pct);
        }
        if (std::getenv("DRS_DEBUG_OCC") && d.OccupancyMaxActiveBlocks) {     // development aid: resident CTAs per SM
            int nb = -1;
            d.OccupancyMaxActiveBlocks(&nb, p->f_sweep, p->spec.nw * 32, (size_t)smem);
            std::fprintf(stderr, "drs: dr_%s: %d CTAs of %d threads per SM (%d registers, %d bytes of shared memory)\n", nm.c_str(), nb,
                         p->spec.nw * 32, p->regs, smem);
        }
    }
    r = d.ModuleGetFunction(&p->f_gold, p->mod, ("gold_" + nm).c_str());
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuModuleGetFunction(gold_): " + cu_err(r));
    r = d.ModuleGetFunction(&p->f_check, p->mod, ("check_" + nm).c_str());
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuModuleGetFunction(check_): " + cu_err(r));
    r = d.ModuleGetFunction(&p->f_signal, p->mod, ("signal_" + nm).c_str());
    if (r == CUDA_SUCCESS) r = d.ModuleGetFunction(&p->f_wait, p->mod, ("wait_" + nm).c_str());
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuModuleGetFunction(signal_/wait_): " + cu_err(r));
    const int prc = load_pair(p);
    if (prc != DRS_OK) return prc;
    if (cudaMalloc(&p->d_fault, sizeof(int)) != cudaSuccess) return fail(DRS_E_CUDA, "cudaMalloc(fault flag)");
    cudaMemset(p->d_fault, 0, sizeof(int));
    if (cudaMalloc(&p->d_res, 2 * sizeof(double)) != cudaSuccess) return fail(DRS_E_CUDA, "cudaMalloc(result)");
    p->loaded = true;
    return load_slab2d(p);
}

int tensor_map_for(drs_plan* p, const void* base, CUtensorMap** out, bool pair = false) {
    std::map<const void*, CUtensorMap>& tmaps = pair ? p->ptmaps : p->tmaps;
    auto it = tmaps.find(base);
    if (it != tmaps.end()) { *out = &it->second; return DRS_OK; }
    const drs::KernelSpec& s = pair ? p->pspec : p->spec;
    if (s.flat != 2 && (reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(DRS_E_ARG, "device buffers must be 16-byte aligned");
    CUtensorMap m;
    if (s.flat == 2) {
        // the kernel fills its stages with cp.async and uses no tensor map: the parameter slot carries zeros
        std::memset(&m, 0, sizeof m);
    } else {
        const CUtensorMapDataType dt = s.dtype == DRS_F64 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
        const cuuint64_t es = (cuuint64_t)s.esize(), L = p->st.L, M = p->st.M, N = p->st.N;
        // L2 promotion of the TMA fetches: 256 B for plane boxes (c5 1536^3: 9.54 -> 9.40 ms, c4 +0.5 %; none / 64 B /
        // 128 B are equal), 128 B for row boxes (2D: no difference).  DRS_TMA_L2PROMO=0..3 overrides (development aid).
        CUtensorMapL2promotion promo = s.dim == 3 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
        if (const char* e = getenv("DRS_TMA_L2PROMO")) promo = (CUtensorMapL2promotion)atoi(e);
        // 2D: rows of N elements, boxes of wb() x rb; 3D: planes of M rows, boxes of wb() x box_rows() x 1
        cuuint32_t rank = s.dim;
        cuuint64_t dims[3] = {N, M, L}, strides[2] = {N * es, N * M * es};
        cuuint32_t box[3] = {(cuuint32_t)s.wb(), (cuuint32_t)(s.dim == 3 ? s.box_rows() : s.rb), 1};
        const cuuint32_t estr[3] = {1, 1, 1};
        if (s.flat == 1) {
            // the whole array as one row of a {total, 1} tensor; a tile arrives as one box of wb() + vec() elements per
            // row, each starting on a 16-byte boundary (a rank-1 map is not an option: the encoder wants a stride array)
            rank = 2;
            dims[0] = L * M * N; dims[1] = 1;
            strides[0] = (dims[0] * es + 15) / 16 * 16;
            box[0] = (cuuint32_t)(s.wb() + s.vec()); box[1] = 1;
        }
        const CUresult r = driver().TensorMapEncodeTiled(&m, dt, rank, const_cast<void*>(base), dims, strides, box, estr,
                                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                                         promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuTensorMapEncodeTiled: " + cu_err(r));
    }
    if (tmaps.size() > 64) tmaps.clear();
    auto ins = tmaps.emplace(base, m);
    *out = &ins.first->second;
    return DRS_OK;
}

struct SlowRange { long long lo, hi; };   // output range along the slow axis, local indices

// ring = frozen ring width of this launch (spec.halo, or the sub-step's share of it);
// sub  = restrict the launch to these slow-axis outputs (time-skewed blocks of drs_run_host)
// seq_off >= 0: this launch is sweep number seq_off of a drs_run_slab call and handles its own step flags
// spec: the specialisation the launch runs (default: the plan's main one; the exact pair kernel has its own tile)
void fill_params(const drs_plan* p, const void* in, void* out, DevParams& q, int ring = -1, const SlowRange* sub = nullptr,
                 int seq_off = -1, const drs::KernelSpec* spec = nullptr) {
    const drs::KernelSpec& s = spec ? *spec : p->spec;
    std::memset(&q, 0, sizeof q);
    q.in = in; q.out = out;
    q.L = p->st.L; q.M = p->st.M; q.N = p->st.N;
    q.halo = ring >= 0 ? ring : s.halo;
    const long long slow = p->local_slow();
    if (!p->slab) { q.slow_lo = q.halo; q.slow_hi = slow - q.halo; }
    else {
        const long long ghost = p->ghost(), org = p->lo - ghost;  // global index of local plane 0
        const long long glo = std::max<long long>(p->lo, s.halo), ghi = std::min<long long>(p->hi, p->g_slow - s.halo);
        q.slow_lo = glo - org; q.slow_hi = ghi - org;
        int b = -1;
        if (out == p->my_bases[0]) b = 0; else if (out == p->my_bases[1]) b = 1;
        if (b >= 0 && p->lower_bases[b] && p->lo > 0) {
            q.peer_lo = p->lower_bases[b];
            q.push_lo0 = p->lo - org; q.push_lo1 = p->lo + ghost - org;
            q.peer_lo_shift = org - (p->lower_lo - ghost);
        }
        if (b >= 0 && p->upper_bases[b] && p->hi < p->g_slow) {
            q.peer_hi = p->upper_bases[b];
            q.push_hi0 = p->hi - ghost - org; q.push_hi1 = p->hi - org;
            q.peer_hi_shift = org - (p->upper_lo - ghost);
        }
    }
    if (sub) { q.slow_lo = std::max(q.slow_lo, sub->lo); q.slow_hi = std::min(q.slow_hi, sub->hi); }
    if (q.slow_hi < q.slow_lo) q.slow_hi = q.slow_lo;
    const long long a0 = (q.halo / s.vec()) * s.vec();
    const long long xspan = std::max<long long>(0, (q.N - q.halo) - a0);
    q.nxs = (int)((xspan + s.wu() - 1) / s.wu());
    const long long nslow = (q.slow_hi - q.slow_lo + s.chunk - 1) / s.chunk;
    if (s.dim == 2) { q.nys = (int)nslow; q.nzs = 1; }
    else {
        const long long yspan = std::max<long long>(0, q.M - 2 * q.halo);
        q.nys = (int)((yspan + s.tile_rows_useful() - 1) / s.tile_rows_useful());
        q.nzs = (int)nslow;
    }
    q.chunk = s.chunk;
    q.fault = p->d_fault;
    if (seq_off >= 0 && p->slab && p->my_flags && p->d_sync && !sub && (q.peer_lo || q.peer_hi)) {
        q.my_flags = (const long long*)p->my_flags;
        q.lower_flag = q.peer_lo ? (long long*)p->lower_flag : nullptr;
        q.upper_flag = q.peer_hi ? (long long*)p->upper_flag : nullptr;
        q.seq_base = (const long long*)p->d_sync;
        q.face_cnt = (unsigned int*)((char*)p->d_sync + sizeof(long long));
        q.seq_off = seq_off;
        // a chunk [za, zb) belongs to a face when it reads that neighbour's ghost planes (rows in 2D) or produces
        // planes that are pushed to it.  The pushed planes are the `ghost` owned planes next to the face, and the input
        // reaches at most `ghost` planes beyond the outputs (Halo for a single sweep; 2 * Halo for a pair launch, which
        // only runs on slabs with ghost = 2 * Halo), so both fall below 2 * ghost.  The chunks are the nzs plane chunks
        // in 3D, the nys row chunks in 2D (one unit = one warp, nxs of them per row chunk).
        const long long ghost = p->ghost(), local = p->local_slow();
        q.face_lo_end = 2 * ghost;
        q.face_hi_begin = local - 2 * ghost;
        const long long units_per_chunk = s.dim == 2 ? (long long)q.nxs
                                          : s.share3d ? (long long)s.nw * ((q.nxs + s.sx - 1) / s.sx) * ((q.nys + s.sy - 1) / s.sy)
                                                      : (long long)q.nxs * q.nys;
        const long long nchunks = s.dim == 2 ? q.nys : q.nzs;
        int nlo = 0, nhi = 0;
        for (long long zc = 0; zc < nchunks; ++zc) {
            const long long za = q.slow_lo + zc * s.chunk, zb = std::min(za + s.chunk, q.slow_hi);
            if (q.lower_flag && za < q.face_lo_end) ++nlo;
            if (q.upper_flag && zb > q.face_hi_begin) ++nhi;
        }
        // the kernel lists the lower-face chunks first, then the upper-face ones; a chunk that touches both
        // faces (thin slabs) is counted on both and keeps its place in the prefix
        q.face_lo_chunks = nlo;
        q.face_hi_chunks = std::min<long long>(nhi, nchunks - nlo);
        q.face_lo_units = (unsigned int)(nlo * units_per_chunk);
        q.face_hi_units = (unsigned int)(nhi * units_per_chunk);
    }
}

int launch_gold(drs_plan* p, const void* in, void* out, cudaStream_t stream) {
    DevParams q;
    fill_params(p, in, out, q);
    void* args[] = {&q};
    unsigned bx = 32, by = 8, bz = 1;
    unsigned gx = (unsigned)((q.N + bx - 1) / bx), gy = (unsigned)((q.M + by - 1) / by), gz = (unsigned)q.L;
    CUresult r = driver().LaunchKernel(p->f_gold, gx, gy, gz, bx, by, bz, 0, (CUstream)stream, args, nullptr);
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "launch gold_: " + cu_err(r));
    p->launches++;
    return DRS_OK;
}

int launch_one(drs_plan* p, const void* in, void* out, cudaStream_t stream, int ring, const SlowRange* sub = nullptr,
               int seq_off = -1);

// `--fuse reuse` (drs_reuse.cuh): the reference's launch shape -- overlapped tiles of bx x by threads, one block
// per tile and chunk of `sn` slow-axis outputs (codegen_2d.hpp:585-598, codegen.hpp:566-571)
int launch_reuse(drs_plan* p, const void* in, void* out, cudaStream_t stream) {
    const drs::KernelSpec& s = p->spec;
    DevParams q;
    fill_params(p, in, out, q);
    void* args[] = {&q};
    const long long H = s.halo;
    const long long nslow = (q.slow_hi - q.slow_lo + s.chunk - 1) / s.chunk;
    if (nslow <= 0 || q.N <= 2 * H) return DRS_OK;
    const unsigned gx = (unsigned)((q.N - 2 * H + (s.rbx - 2 * H) - 1) / (s.rbx - 2 * H));
    unsigned gy, gz;
    if (s.dim == 3) {
        if (q.M <= 2 * H) return DRS_OK;
        gy = (unsigned)((q.M - 2 * H + (s.rby - 2 * H) - 1) / (s.rby - 2 * H));
        gz = (unsigned)nslow;
    } else { gy = (unsigned)nslow; gz = 1; }
    if (gy > 65535u || gz > 65535u) return fail(DRS_E_ARG, "grid too large for the data-reuse mode: raise --sn");
    CUresult r = driver().LaunchKernel(p->f_sweep, gx, gy, gz, (unsigned)s.rbx, (unsigned)s.rby, 1, 0, (CUstream)stream, args, nullptr);
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "launch dr_ (data reuse): " + cu_err(r));
    p->launches++;
    return DRS_OK;
}

int launch_sweep(drs_plan* p, const void* in, void* out, cudaStream_t stream) {
    if (in == out) return fail(DRS_E_ARG, "d_in and d_out must differ");
    if (p->spec.reuse) return launch_reuse(p, in, out, stream);
    if (!p->spec.tma_ok) return launch_gold(p, in, out, stream);
    const int T = p->spec.sub_launches;
    if (T <= 1) return launch_one(p, in, out, stream, -1);
    // sub-step s (1..T) advances [s*r, dim - s*r) from the previous level; levels in between live in
    // scratch buffers whose rings are never read
    const size_t bytes = (size_t)p->st.L * p->st.M * p->st.N * p->spec.esize();
    for (int i = 0; i < (T > 2 ? 2 : 1); ++i)
        if (!p->scratch[i] && cudaMalloc(&p->scratch[i], bytes) != cudaSuccess)
            return fail(DRS_E_CUDA, "cudaMalloc of the temporal scratch buffer failed");
    const void* src = in;
    for (int s = 1; s <= T; ++s) {
        void* dst = s == T ? out : p->scratch[(s - 1) & 1];
        int rc = launch_one(p, src, dst, stream, s * p->spec.base_order);
        if (rc != DRS_OK) return rc;
        src = dst;
    }
    return DRS_OK;
}

int launch_one(drs_plan* p, const void* in, void* out, cudaStream_t stream, int ring, const SlowRange* sub, int seq_off) {
    CUtensorMap* tm = nullptr;
    int rc = tensor_map_for(p, in, &tm);
    if (rc != DRS_OK) return rc;
    // 128-bit stores: a misaligned destination would be a sticky device fault, not an error code
    if (!p->spec.flat && (reinterpret_cast<uintptr_t>(out) & 15) != 0) return fail(DRS_E_ARG, "device buffers must be 16-byte aligned");
    DevParams q;
    fill_params(p, in, out, q, ring, sub, seq_off);
    const long long tiles = (long long)q.nxs * q.nys * q.nzs;
    if (tiles <= 0) return DRS_OK;
    const long long ctas = p->spec.ctas(q.nxs, q.nys, q.nzs);
    if (ctas > 0x7fffffffLL) return fail(DRS_E_ARG, "grid too large");
    void* args[] = {tm, &q};
    // 3D: drslab_ runs the flagged sweeps of drs_run_slab (dr_ makes the peer stores itself).  2D: dr_ makes none, so
    // every launch of a slab plan with peers runs drslab_ (flags or not); without peers the ghost rows stay frozen.
    const bool slab_fn = p->spec.dim == 2 ? p->slab && p->my_bases[0] != nullptr : q.my_flags != nullptr;
    if (slab_fn && !p->f_slab) return fail(DRS_E_ARG, "this plan has no slab kernel");
    CUresult r = driver().LaunchKernel(slab_fn ? p->f_slab : p->f_sweep, (unsigned)ctas, 1, 1, (unsigned)(p->spec.nw * 32), 1, 1,
                                       (unsigned)p->spec.smem_bytes(), (CUstream)stream, args, nullptr);
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, std::string(slab_fn ? "launch drslab_: " : "launch dr_: ") + cu_err(r));
    p->launches++;
    return DRS_OK;
}

// One exact pair launch (kernels/pair/drs_pair3d.cuh, kernels/pair2d/drs_pair2d.cuh): two sweeps of drs_run's ping-pong
// schedule, from the level in `in` to the level two steps later in the interior of `out`.  a / b are the run's buffers:
// even levels have a's ring, odd ones b's.  One CTA per tile in 3D, NW warp tiles per CTA in 2D (pspec.ctas).
// sub: store only these slow-axis outputs (time-skewed blocks of drs_run_host; DESIGN 3.6 for what the chunks read).
int launch_pair(drs_plan* p, const void* in, void* out, const void* a, const void* b, cudaStream_t stream,
                const SlowRange* sub = nullptr) {
    if (in == out) return fail(DRS_E_ARG, "d_in and d_out must differ");
    CUtensorMap* tm = nullptr;
    int rc = tensor_map_for(p, in, &tm, true);
    if (rc != DRS_OK) return rc;
    CUtensorMap map_in = *tm;          // (the next lookup may clear the cache)
    rc = tensor_map_for(p, a, &tm, true);
    if (rc != DRS_OK) return rc;
    CUtensorMap map_a = *tm;
    if ((reinterpret_cast<uintptr_t>(out) & 15) != 0) return fail(DRS_E_ARG, "device buffers must be 16-byte aligned");
    DevParams q;
    fill_params(p, in, out, q, -1, sub, -1, &p->pspec);
    const long long tiles = (long long)q.nxs * q.nys * q.nzs;
    if (tiles <= 0) return DRS_OK;
    const long long ctas = p->pspec.ctas(q.nxs, q.nys, q.nzs);
    if (ctas > 0x7fffffffLL) return fail(DRS_E_ARG, "grid too large");
    const void* ring_a = a;
    const void* ring_b = b;
    void* args[] = {&map_in, &map_a, &q, &ring_a, &ring_b};
    CUresult r = driver().LaunchKernel(p->f_pair, (unsigned)ctas, 1, 1, (unsigned)(p->pspec.nw * 32), 1, 1,
                                       (unsigned)p->pspec.smem_bytes(), (CUstream)stream, args, nullptr);
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "launch drpair_: " + cu_err(r));
    p->launches++;
    return DRS_OK;
}

// One pair launch of a pair slab (kernels/slabpair/drs_slabpair3d.cuh): the pair of sweeps of drs_run_slab's launch
// `seq_off` (< 0: no step flags), from the level in `in` to the level two steps later on the owned output planes of
// `out`, pushed to the neighbours' deep ghost planes.  Level 0's global ring is A's (my_bases[0]), level 1's is B's.
int launch_slabpair(drs_plan* p, const void* in, void* out, cudaStream_t stream, int seq_off) {
    if (in == out) return fail(DRS_E_ARG, "d_in and d_out must differ");
    if (!p->f_slabpair) return fail(DRS_E_ARG, "this plan has no slab pair kernel");
    const void* a = p->my_bases[0];
    CUtensorMap* tm = nullptr;
    int rc = tensor_map_for(p, in, &tm, true);
    if (rc != DRS_OK) return rc;
    CUtensorMap map_in = *tm;          // (the next lookup may clear the cache)
    rc = tensor_map_for(p, a, &tm, true);
    if (rc != DRS_OK) return rc;
    CUtensorMap map_a = *tm;
    if ((reinterpret_cast<uintptr_t>(out) & 15) != 0) return fail(DRS_E_ARG, "device buffers must be 16-byte aligned");
    DevParams q;
    fill_params(p, in, out, q, -1, nullptr, seq_off, &p->pspec);
    const long long tiles = (long long)q.nxs * q.nys * q.nzs;
    if (tiles <= 0) return DRS_OK;
    if (tiles > 0x7fffffffLL) return fail(DRS_E_ARG, "grid too large");
    const void* ring_a = a;
    const void* ring_b = p->my_bases[1];
    // the global ring planes [0, Halo) and [G - Halo, G) in local coordinates, clamped to the array
    const long long org = p->lo - p->ghost(), H = p->spec.halo, L = p->st.L;
    int ring_lo = (int)std::min(L, std::max(0LL, H - org));
    int ring_hi = (int)std::min(L, std::max(0LL, p->g_slow - H - org));
    void* args[] = {&map_in, &map_a, &q, &ring_a, &ring_b, &ring_lo, &ring_hi};
    CUresult r = driver().LaunchKernel(p->f_slabpair, (unsigned)tiles, 1, 1, (unsigned)(p->pspec.nw * 32), 1, 1,
                                       (unsigned)p->pspec.smem_bytes(), (CUstream)stream, args, nullptr);
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "launch drslabpair_: " + cu_err(r));
    p->launches++;
    return DRS_OK;
}

// The slab step-flag kernels (drs_gold.cuh): signal_ release-stores `value` into the non-null remote flag words;
// wait_ waits until the selected words of `flags` (lower, upper) hold >= value, or sets the fault flag after 5 s.
int launch_signal(drs_plan* p, cudaStream_t stream, void* lower, void* upper, long long value) {
    void* args[] = {&lower, &upper, &value};
    CUresult r = driver().LaunchKernel(p->f_signal, 1, 1, 1, 32, 1, 1, 0, (CUstream)stream, args, nullptr);
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "launch signal_: " + cu_err(r));
    p->launches++;
    return DRS_OK;
}

int launch_wait(drs_plan* p, cudaStream_t stream, const void* flags, int lo, int hi, long long value) {
    void* args[] = {(void*)&flags, &lo, &hi, &value, &p->d_fault};
    CUresult r = driver().LaunchKernel(p->f_wait, 1, 1, 1, 32, 1, 1, 0, (CUstream)stream, args, nullptr);
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "launch wait_: " + cu_err(r));
    p->launches++;
    return DRS_OK;
}

// Whether drs_run runs pair launches on this plan.  Not on a slab: the pair kernel takes its ring from the local
// array's edges instead of the global faces, and it makes no peer stores.
bool uses_pairs(const drs_plan* p) { return p->pair && !p->slab; }

// drs_run's n sweeps over (a, b): sweep s writes the interior of bufs[(s+1)%2] from bufs[s%2].  Plans with exact pair
// launches run p pairs (pair i: bufs[i%2] -> level 2i+2 in bufs[(i+1)%2]) and then s single sweeps (generate.hpp:
// pair_split); both buffers end exactly as after n single sweeps.
int enqueue_run(drs_plan* p, void* a, void* b, int n, cudaStream_t stream) {
    int pairs = 0, singles = n;
    if (uses_pairs(p)) drs::pair_split(n, pairs, singles);
    int rc = DRS_OK;
    for (int i = 0; i < pairs && rc == DRS_OK; ++i)
        rc = (i & 1) ? launch_pair(p, b, a, a, b, stream) : launch_pair(p, a, b, a, b, stream);
    for (int s = 0; s < singles && rc == DRS_OK; ++s)
        rc = (s & 1) ? launch_sweep(p, b, a, stream) : launch_sweep(p, a, b, stream);
    return rc;
}

int check_sizes(const drs::Stencil& st) {
    if (st.M <= 0 || st.N <= 0 || (st.dim == 3 && st.L <= 0)) return fail(DRS_E_ARG, "grid extents must be positive");
    if (st.M > 0x7fffff00LL || st.N > 0x7fffff00LL || st.L > 0x7fffff00LL) return fail(DRS_E_ARG, "extent too large");
    return DRS_OK;
}

int make_plan(const drs_stencil* s, const drs_knobs* k, drs_plan** out, bool compile) {
    if (!s || !k || !out) return fail(DRS_E_ARG, "null argument");
    int rc = check_sizes(s->st);
    if (rc != DRS_OK) return rc;
    drs_plan* p = new drs_plan();
    p->st = s->st;
    p->knobs = *k;
    p->spec.name = s->name;
    std::string err = drs::choose_spec(s->st, *k, p->spec);
    if (!err.empty()) {
        delete p;
        // `--fuse reuse` refuses what the reference refuses, with its messages (drstencil_2d.hpp:217-220, codegen_2d.hpp:52-56)
        if (err.rfind("NOREUSE:", 0) == 0) return fail(DRS_E_NOREUSE, err.substr(8));
        if (err.rfind("CONFIG:", 0) == 0) return fail(DRS_E_CONFIG, err.substr(7));
        return fail(DRS_E_ARG, err);
    }
    p->source = drs::generate_tu(p->spec);
    p->pair = drs::pair_spec(p->st, p->spec, p->pspec);
    if (p->pair) p->pair_source = drs::generate_pair_tu(p->pspec);
    if (compile) {
        rc = compile_cubin(p->source, p->cubin, p->cache_key);
        if (rc == DRS_OK && p->pair) rc = compile_cubin(p->pair_source, p->pair_cubin, p->pair_key, Unit::PAIR);
        if (rc != DRS_OK) { delete p; return rc; }
    }
    *out = p;
    return DRS_OK;
}

}  // namespace

extern "C" {

void drs_knobs_default(drs_knobs* k) {
    std::memset(k, 0, sizeof *k);
    k->step = 1; k->dist = 0; k->streaming = 0; k->bx = 16; k->by = 16; k->sn = 16; k->stream_unroll = 4;
    k->block_merge_x = k->block_merge_y = k->cyclic_merge_x = k->cyclic_merge_y = 1;
    k->prefetch = 0; k->merge_forward = 5; k->check = 0;
    k->dtype = DRS_F64; k->fuse = DRS_FUSE_TEMPORAL; k->explicit_mask = 0;
}

int drs_stencil_from_file(const char* path, int is3d, drs_stencil** out) {
    if (!path || !out) return fail(DRS_E_ARG, "null argument");
    drs_stencil* s = new drs_stencil();
    if (!s->st.read_stc(path, is3d != 0)) {
        delete s;
        return fail(DRS_E_IO, "Error opening stencil file.");
    }
    // kernel name = file name minus its last four characters, as main.cpp:243-244 (directory dropped)
    std::string nm = path;
    size_t sl = nm.rfind('/');
    if (sl != std::string::npos) nm = nm.substr(sl + 1);
    if (nm.size() > 4) nm.erase(nm.size() - 4);
    for (char& c : nm) if (!(isalnum((unsigned char)c) || c == '_')) c = '_';
    if (nm.empty()) nm = "stencil";
    s->name = nm;
    *out = s;
    return DRS_OK;
}

int drs_stencil_from_points(int dim, const int* offsets, const double* coefs, int npoints, long long L, long long M,
                            long long N, int iterations, drs_stencil** out) {
    if ((dim != 2 && dim != 3) || !offsets || !coefs || npoints <= 0 || !out) return fail(DRS_E_ARG, "bad stencil description");
    drs_stencil* s = new drs_stencil();
    s->st.set_points(dim, offsets, coefs, npoints);
    s->st.L = dim == 3 ? L : 1; s->st.M = M; s->st.N = N; s->st.iterations = iterations;
    *out = s;
    return DRS_OK;
}

void drs_stencil_destroy(drs_stencil* s) { delete s; }

int drs_stencil_set_name(drs_stencil* s, const char* name) {
    if (!s || !name || !*name) return fail(DRS_E_ARG, "bad name");
    std::string nm = name;
    for (char& c : nm) if (!(isalnum((unsigned char)c) || c == '_')) c = '_';
    s->name = nm;
    return DRS_OK;
}

int drs_stencil_set_size(drs_stencil* s, long long L, long long M, long long N, int iterations) {
    if (!s) return fail(DRS_E_ARG, "null stencil");
    s->st.L = s->st.dim == 3 ? L : 1; s->st.M = M; s->st.N = N; s->st.iterations = iterations;
    return DRS_OK;
}

int drs_stencil_compose(drs_stencil* s, int step) {
    if (!s || step < 1) return fail(DRS_E_ARG, "step must be >= 1");
    s->st.compose(step);
    return DRS_OK;
}

int drs_stencil_size(const drs_stencil* s, long long dims[3], int* iterations) {
    if (!s) return fail(DRS_E_ARG, "null stencil");
    if (dims) { dims[0] = s->st.L; dims[1] = s->st.M; dims[2] = s->st.N; }
    if (iterations) *iterations = s->st.iterations;
    return DRS_OK;
}

int drs_stencil_terms(const drs_stencil* s, int* offsets3, double* coefs, int capacity) {
    if (!s) return fail(DRS_E_ARG, "null stencil");
    std::vector<drs::Term> t = s->st.terms();
    if (offsets3 && coefs) {
        if (capacity < (int)t.size()) return fail(DRS_E_ARG, "buffer too small");
        for (size_t q = 0; q < t.size(); ++q) {
            offsets3[3 * q] = t[q].dk; offsets3[3 * q + 1] = t[q].dj; offsets3[3 * q + 2] = t[q].di;
            coefs[q] = t[q].coef;
        }
    }
    return (int)t.size();
}

int drs_stencil_term_text(const drs_stencil* s, int q, char* buf, size_t buflen) {
    if (!s || !buf || buflen == 0) return fail(DRS_E_ARG, "null argument");
    if (q < 0 || q >= (int)s->st.points.size()) return fail(DRS_E_ARG, "term index out of range");
    auto it = s->st.points.begin();
    std::advance(it, q);
    std::snprintf(buf, buflen, "%s", drs::coef_literal_text(it->second).c_str());
    return DRS_OK;
}

int drs_stencil_analyze(const drs_stencil* s, int dist, int merge_forward, int* halo, int* dist_out, int* range,
                        int sizes[4]) {
    if (!s) return fail(DRS_E_ARG, "null stencil");
    drs::Analysis a;
    const bool ok = s->st.analyze(dist, merge_forward, a);
    if (halo) *halo = a.halo;
    if (dist_out) *dist_out = a.dist;
    if (sizes) {
        sizes[0] = (int)a.forward_slow.size(); sizes[1] = (int)a.forward_mid.size();
        sizes[2] = (int)a.forward_fast.size(); sizes[3] = (int)a.backward.size();
    }
    if (!ok) return fail(DRS_E_NOREUSE, "No data to reuse. You can try another dist.");
    if (range) *range = a.range();
    return DRS_OK;
}

int drs_plan_create(const drs_stencil* s, const drs_knobs* k, drs_plan** out) { return make_plan(s, k, out, true); }

int drs_plan_warm_cache(const drs_stencil* s, const drs_knobs* k) {
    drs_plan* p = nullptr;
    int rc = make_plan(s, k, &p, true);
    if (rc == DRS_OK) delete p;
    return rc;
}

void drs_plan_destroy(drs_plan* p) {
    if (!p) return;
    if (p->loaded) {
        cudaFree(p->d_fault);
        cudaFree(p->d_res);
        for (void* b : p->h_dev) if (b) cudaFree(b);
        for (void* b : p->scratch) if (b) cudaFree(b);
        if (p->d_sync) cudaFree(p->d_sync);
        for (cudaStream_t st : {p->hs_up, p->hs_run, p->hs_dn, p->cap_stream}) if (st) cudaStreamDestroy(st);
        for (auto& g : p->graphs) cudaGraphExecDestroy(g.second.exec);
        if (p->mod) driver().ModuleUnload(p->mod);
        for (auto& m : p->pmods) driver().ModuleUnload(m.second.first);
        if (p->smod) driver().ModuleUnload(p->smod);
        if (p->spmod) driver().ModuleUnload(p->spmod);
    }
    delete p;
}

int drs_plan_get_info(const drs_plan* p, drs_plan_info* info) {
    if (!p || !info) return fail(DRS_E_ARG, "null argument");
    std::memset(info, 0, sizeof *info);
    const drs::KernelSpec& s = p->spec;
    info->dim = s.dim; info->dtype = s.dtype; info->step = s.step; info->fuse = s.fuse;
    info->L = p->st.L; info->M = p->st.M; info->N = p->st.N;
    info->halo = s.halo; info->npoints = (int)s.chain.size(); info->timesteps_per_sweep = s.step;
    info->warps_per_cta = s.nw; info->tile_x = s.wu(); info->tile_y = s.dim == 3 ? s.tile_rows_useful() : 1;
    info->chunk = s.chunk; info->stages = s.st; info->rows_per_stage = s.dim == 2 ? s.rb : 1;
    DevParams q;
    fill_params(p, nullptr, nullptr, q);
    const long long tiles = (long long)q.nxs * q.nys * q.nzs;
    info->grid_x = (int)(tiles > 0 ? s.ctas(q.nxs, q.nys, q.nzs) : 0); info->grid_y = 1; info->grid_z = 1;
    info->block = s.nw * 32;
    info->smem_bytes = s.tma_ok ? s.smem_bytes() : 0;
    info->regs_per_thread = p->regs; info->spill_bytes = p->spill;
    // computed / useful points
    const double useful = (double)std::max<long long>(1, q.N - 2 * s.halo) * (double)std::max<long long>(1, q.slow_hi - q.slow_lo) *
                          (s.dim == 3 ? (double)std::max<long long>(1, q.M - 2 * s.halo) : 1.0);
    double computed;
    if (s.dim == 2) computed = (double)q.nxs * s.wt() * ((double)(q.slow_hi - q.slow_lo) + (double)q.nys * s.ts * (2 * s.rj + 1));
    else computed = (double)q.nxs * s.wt() * (double)q.nys * s.tile_rows() *
                    ((double)(q.slow_hi - q.slow_lo) + (s.fused3d ? (double)q.nzs * (2 * s.ts * s.rk + s.ts - 1) : 0.0));
    info->redundancy = computed / useful;
    std::snprintf(info->kernel_name, sizeof info->kernel_name, "%s%s", (s.tma_ok || s.reuse) ? "dr_" : "gold_", s.name.c_str());
    if (s.reuse) {
        info->warps_per_cta = (s.rbx * s.rby + 31) / 32; info->tile_x = s.rbx - 2 * s.halo; info->tile_y = s.dim == 3 ? s.rby - 2 * s.halo : 1;
        info->block = s.rbx * s.rby; info->stages = 0; info->smem_bytes = 0;
        info->redundancy = (double)s.rbx / std::max(1, s.rbx - 2 * s.halo) * (s.dim == 3 ? (double)s.rby / std::max(1, s.rby - 2 * s.halo) : 1.0);
    }
    return DRS_OK;
}

const char* drs_plan_source(const drs_plan* p) { return p ? p->source.c_str() : ""; }
const char* drs_plan_note(const drs_plan* p) { return p ? p->spec.note.c_str() : ""; }
const char* drs_plan_cache_key(const drs_plan* p) { return p ? p->cache_key.c_str() : ""; }
const char* drs_plan_pair_source(const drs_plan* p) { return p ? p->pair_source.c_str() : ""; }
const char* drs_plan_pair_cache_key(const drs_plan* p) { return p ? p->pair_key.c_str() : ""; }
const char* drs_plan_slab_source(const drs_plan* p) { return p ? p->slab_source.c_str() : ""; }
const char* drs_plan_slab_cache_key(const drs_plan* p) { return p ? p->slab_key.c_str() : ""; }
const char* drs_plan_slab_pair_source(const drs_plan* p) { return p ? p->slabpair_source.c_str() : ""; }
const char* drs_plan_slab_pair_cache_key(const drs_plan* p) { return p ? p->slabpair_key.c_str() : ""; }

int drs_sweep(drs_plan* p, const void* d_in, void* d_out, void* stream) {
    if (!p || !d_in || !d_out) return fail(DRS_E_ARG, "null argument");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    return launch_sweep(p, d_in, d_out, (cudaStream_t)stream);
}

int drs_gold_sweep(drs_plan* p, const void* d_in, void* d_out, void* stream) {
    if (!p || !d_in || !d_out) return fail(DRS_E_ARG, "null argument");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    return launch_gold(p, d_in, d_out, (cudaStream_t)stream);
}

static void drop_graphs(drs_plan* p) {
    for (auto& g : p->graphs) cudaGraphExecDestroy(g.second.exec);
    p->graphs.clear();
}

// A launch sequence as an instantiated CUDA graph: built once per key by capturing the very same
// cuLaunchKernel calls (enqueue(stream)) on a private stream, replayed with one cudaGraphLaunch.  Saves the
// per-launch gap between dependent kernels, which is what separates a 45 us sweep (c1: 4096^2) from the
// roofline (47.2 -> 45.4 us per sweep on B200).  Returns false when the caller must launch directly: graphs
// are off, the caller is capturing `stream` itself, a tensor map cannot be encoded, or anything about the
// capture fails (which switches graphs off for the plan).
static bool run_graph(drs_plan* p, void* a, void* b, int n, bool slab, cudaStream_t stream,
                      const std::function<int(cudaStream_t)>& enqueue) {
    if (!p->use_graph) return false;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cs) != cudaSuccess) { cudaGetLastError(); return false; }
    if (cs != cudaStreamCaptureStatusNone) return false;
    const auto key = std::make_tuple((const void*)a, (const void*)b, n, slab);
    auto it = p->graphs.find(key);
    if (it == p->graphs.end()) {
        if (!p->cap_stream && cudaStreamCreateWithFlags(&p->cap_stream, cudaStreamNonBlocking) != cudaSuccess) {
            cudaGetLastError(); p->use_graph = false; return false;
        }
        // tensor maps are encoded outside the capture (host-only, but keeps the captured region to launches);
        // pair launches run in drs_run's sequence on plain plans and in drs_run_slab's on pair slabs
        CUtensorMap* tm = nullptr;
        if (tensor_map_for(p, a, &tm) != DRS_OK || tensor_map_for(p, b, &tm) != DRS_OK) return false;
        if ((slab ? p->slab_pairs : uses_pairs(p)) &&
            (tensor_map_for(p, a, &tm, true) != DRS_OK || tensor_map_for(p, b, &tm, true) != DRS_OK)) return false;
        const long long l0 = p->launches;
        if (cudaStreamBeginCapture(p->cap_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError(); p->use_graph = false; return false;
        }
        const int rc = enqueue(p->cap_stream);
        cudaGraph_t g = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(p->cap_stream, &g);
        const int kernels = (int)(p->launches - l0);
        p->launches = l0;                                       // captured, not run
        cudaGraphExec_t exec = nullptr;
        if (rc != DRS_OK || ce != cudaSuccess || !g || cudaGraphInstantiate(&exec, g, 0) != cudaSuccess) {
            if (g) cudaGraphDestroy(g);
            cudaGetLastError(); p->use_graph = false; return false;
        }
        cudaGraphDestroy(g);
        if (p->graphs.size() >= 16) drop_graphs(p);
        it = p->graphs.emplace(key, drs_plan::RunGraph{exec, kernels}).first;
    }
    if (cudaGraphLaunch(it->second.exec, stream) != cudaSuccess) { cudaGetLastError(); p->use_graph = false; return false; }
    p->launches += it->second.kernels;
    return true;
}

// Sweeps of a run of `iterations` timesteps: the ping-pong loop always runs whole pairs, so A ends with the result.
static int sweeps_for(const drs_plan* p, int iterations) {
    int n = 0;
    for (int t = 0; t < iterations; t += 2 * p->spec.step) n += 2;
    return n;
}

static int run_schedule(drs_plan* p, void* a, void* b, int iterations, void* stream, int* sweeps, bool gold) {
    if (!p || !a || !b) return fail(DRS_E_ARG, "null argument");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    const int n = sweeps_for(p, iterations);
    if (gold) {
        for (int s = 0; s < n; ++s) {
            rc = (s & 1) ? launch_gold(p, b, a, (cudaStream_t)stream) : launch_gold(p, a, b, (cudaStream_t)stream);
            if (rc != DRS_OK) return rc;
        }
    } else {
        const bool graph = p->spec.tma_ok && p->spec.sub_launches <= 1 && a != b && n >= 2;
        auto enqueue = [&](cudaStream_t st) { return enqueue_run(p, a, b, n, st); };
        if (!(graph && run_graph(p, a, b, n, false, (cudaStream_t)stream, enqueue)) && (rc = enqueue((cudaStream_t)stream)) != DRS_OK)
            return rc;
    }
    if (sweeps) *sweeps = n;
    return DRS_OK;
}

int drs_plan_pair_split(const drs_plan* p, int iterations, int* pairs, int* singles) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    const int n = sweeps_for(p, iterations);
    int np = 0, ns = n;
    if (uses_pairs(p)) drs::pair_split(n, np, ns);
    if (pairs) *pairs = np;
    if (singles) *singles = ns;
    return n;
}

int drs_plan_set_pairs(drs_plan* p, int enable) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    if (p->slab) return fail(DRS_E_ARG, "a slab plan has its own pair launches (drs_plan_set_slab_pairs)");
    const drs::KernelSpec& s = p->spec;
    drs::KernelSpec ps;
    bool has = false;
    std::string src;
    if (enable) {
        if (s.dim == 2) {
            const std::string why = drs::pair_spec2d(p->st, s, ps);
            if (!why.empty()) return fail(DRS_E_ARG, "no 2D pair kernel for this plan: " + why);
            src = drs::generate_pair2d_tu(ps);
        } else {
            if (s.step != 1 || s.ts != 1 || s.sub_launches > 1)
                return fail(DRS_E_ARG, "pair launches need a step-1 plan (two single steps per launch)");
            if (s.reuse) return fail(DRS_E_ARG, "pair launches are not available with --fuse reuse");
            if (!s.tma_ok) return fail(DRS_E_ARG, "the plan runs the naive kernel (operator too deep for the TMA sweep)");
            if (s.flat) return fail(DRS_E_ARG, "the pair kernel needs a 16-byte row pitch (N a multiple of 2 in fp64, 4 in fp32)");
            if (!drs::pair_spec(p->st, s, ps, false)) return fail(DRS_E_ARG, "no pair kernel for this operator's depth-2 tile");
            src = drs::generate_pair_tu(ps);
        }
        has = true;
    } else if (drs::pair_spec(p->st, s, ps)) {       // the default rule (make_plan)
        src = drs::generate_pair_tu(ps);
        has = true;
    }
    if (has == p->pair && src == p->pair_source) return DRS_OK;
    std::string key;
    std::vector<char> cubin;
    if (has) {
        const int rc = compile_cubin(src, cubin, key, s.dim == 2 ? Unit::PAIR2D : Unit::PAIR);
        if (rc != DRS_OK) return rc;
    }
    drop_graphs(p);          // the graph key (A, B, sweep count, slab) does not include this setting
    p->ptmaps.clear();       // boxes of the new unit's tile
    p->pair = has;
    p->pspec = has ? ps : drs::KernelSpec();
    p->pair_source = std::move(src);
    p->pair_key = std::move(key);
    p->pair_cubin = std::move(cubin);
    return p->loaded ? load_pair(p) : DRS_OK;
}

int drs_run(drs_plan* p, void* d_a, void* d_b, int iterations, void* stream, int* sweeps) {
    return run_schedule(p, d_a, d_b, iterations, stream, sweeps, false);
}
int drs_gold_run(drs_plan* p, void* d_a, void* d_b, int iterations, void* stream, int* sweeps) {
    return run_schedule(p, d_a, d_b, iterations, stream, sweeps, true);
}

int drs_plan_sync_check(drs_plan* p, void* stream) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    if (!p->loaded) return DRS_OK;
    cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("stream sync: ") + cudaGetErrorString(e));
    int f = 0;
    e = cudaMemcpy(&f, p->d_fault, sizeof f, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("fault flag read: ") + cudaGetErrorString(e));
    if (f) {
        cudaMemset(p->d_fault, 0, sizeof(int));
        return fail(DRS_E_KERNEL, f == 2 ? "slab step flag never arrived from a neighbour GPU (5 s watchdog)"
                                         : "sweep kernel pipeline watchdog fired (a TMA stage never arrived)");
    }
    return DRS_OK;
}

// Levels of each launch of a streamed host run of n sweeps: drs_run's launch sequence (pair_split: 2 for a pair
// launch, then the single sweeps' 1s) on plans where drs_run pairs, n single sweeps otherwise.
static std::vector<int> launch_depths(const drs_plan* p, int n) {
    int pairs = 0, singles = n;
    if (uses_pairs(p)) drs::pair_split(n, pairs, singles);
    std::vector<int> depth(pairs, 2);
    depth.insert(depth.end(), singles, 1);
    return depth;
}

// Slow-axis units per block of the streamed host run of launches `depth`, 0 = run the plain copy-sweep-copy
// sequence.  A block must be at least drs::min_block thick (core/host_schedule.hpp: 2 halos, 4 with pair
// launches); blocks of >= 32 MiB keep the copy engines efficient, at most ~16 of them keep the number of small
// launches low.
static long long host_block_units(const drs_plan* p, const std::vector<int>& depth, bool allow_slab = false) {
    const drs::KernelSpec& s = p->spec;
    if (p->host_block < 0 || (p->slab && !allow_slab) || !s.tma_ok || s.sub_launches > 1 || depth.empty()) return 0;
    const long long slow = p->local_slow(), H = s.halo;
    const double unit = (double)(s.dim == 3 ? p->st.M * p->st.N : p->st.N) * s.esize();
    long long S = p->host_block;
    if (S == 0) {
        const double target = std::max(32.0 * 1048576.0, unit * (double)slow / 16.0);
        S = (long long)std::ceil(target / unit);
        S = (S + s.chunk - 1) / s.chunk * s.chunk;     // whole tiles per launch
    }
    S = std::max(S, drs::min_block(depth, H));
    return S < slow ? S : 0;
}

// The emitted main()'s data path (H2D, the ping-pong schedule, D2H) in the time-skewed block order of
// core/host_schedule.hpp: uploads on one stream, launches on a second, downloads on a third, chained
// by events -- the wall time tends to max(H2D, sweeps, D2H) instead of their sum.  Odd launches run
// dA -> dB, even ones dB -> dA; a pair launch takes level 0's ring from dA and level 1's from dB, whose ring
// is the cleared one.  Local plane i is host[i - h0].  clear_b: clear dB before the first launch.
// Face steps (slab runs) use the flag values flag_base + 1 ...: launches that touch a face are bracketed by
// the flag kernels, and the upload that brings a face's level-0 planes is followed by a peer copy of them into
// the neighbour's ghosts.  `what` prefixes the message of a CUDA error found at the end.
static int run_blocks(drs_plan* p, const std::vector<drs::HostStep>& steps, char* dA, char* dB, char* host, long long h0,
                      bool clear_b, long long flag_base, const char* what, float* device_ms) {
    const long long H = p->spec.halo, local = p->local_slow(), org = p->lo - H;
    const size_t unit = (size_t)(p->spec.dim == 3 ? p->st.M * p->st.N : p->st.N) * p->spec.esize();
    for (cudaStream_t* st : {&p->hs_up, &p->hs_run, &p->hs_dn})
        if (!*st && cudaStreamCreateWithFlags(st, cudaStreamNonBlocking) != cudaSuccess)
            return fail(DRS_E_CUDA, "cudaStreamCreate failed");
    int B = 0;
    for (const drs::HostStep& st : steps) B = std::max(B, st.block + 1);
    std::vector<cudaEvent_t> up(B), done(B);
    cudaEvent_t e0, e1, fin;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventCreateWithFlags(&fin, cudaEventDisableTiming);
    for (int b = 0; b < B; ++b) {
        cudaEventCreateWithFlags(&up[b], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming);
    }
    cudaEventRecord(e0, 0);
    for (cudaStream_t st : {p->hs_up, p->hs_run, p->hs_dn}) cudaStreamWaitEvent(st, e0, 0);
    // every upload is queued first: the copy engine runs ahead of the sweeps as far as it can
    int rc = DRS_OK;
    for (const drs::HostStep& st : steps) {
        if (st.kind != drs::HostStep::UPLOAD || rc != DRS_OK) continue;
        cudaMemcpyAsync(dA + st.lo * unit, host + (st.lo - h0) * unit, (size_t)(st.hi - st.lo) * unit, cudaMemcpyHostToDevice, p->hs_up);
        if ((st.faces & drs::INIT_LOWER) && p->lower_bases[0]) {
            // my planes [H, 2H) are the lower neighbour's upper ghost: same plane shift as the kernel's push
            const long long shift = org - (p->lower_lo - H);
            cudaMemcpyAsync((char*)p->lower_bases[0] + (H + shift) * unit, dA + H * unit, (size_t)H * unit, cudaMemcpyDefault, p->hs_up);
            rc = launch_signal(p, p->hs_up, p->lower_flag, nullptr, flag_base + 1);
        }
        if ((st.faces & drs::INIT_UPPER) && p->upper_bases[0] && rc == DRS_OK) {
            const long long shift = org - (p->upper_lo - H);
            cudaMemcpyAsync((char*)p->upper_bases[0] + (local - 2 * H + shift) * unit, dA + (local - 2 * H) * unit, (size_t)H * unit,
                            cudaMemcpyDefault, p->hs_up);
            rc = launch_signal(p, p->hs_up, nullptr, p->upper_flag, flag_base + 1);
        }
        cudaEventRecord(up[st.block], p->hs_up);
    }
    // the reference's h_out is all zeros (getZero2DArray); only its frozen ring is ever read before
    // it is written, and no sweep writes the ring, so one clear serves every later call
    if (clear_b) {
        cudaMemsetAsync(dB, 0, unit * (size_t)local, p->hs_run);
        p->h_dev_b_ring_zero = true;
    }
    for (const drs::HostStep& st : steps) {
        if (rc != DRS_OK) break;
        if (st.kind == drs::HostStep::UPLOAD) {
            cudaStreamWaitEvent(p->hs_run, up[st.block], 0);
        } else if (st.kind == drs::HostStep::PAIR) {
            const SlowRange r = {st.lo, st.hi};
            rc = (st.launch & 1) ? launch_pair(p, dA, dB, dA, dB, p->hs_run, &r) : launch_pair(p, dB, dA, dA, dB, p->hs_run, &r);
        } else if (st.kind == drs::HostStep::SWEEP) {
            if (st.faces & (drs::WAIT_LOWER | drs::WAIT_UPPER))
                rc = launch_wait(p, p->hs_run, p->my_flags, (st.faces & drs::WAIT_LOWER) != 0, (st.faces & drs::WAIT_UPPER) != 0,
                                 flag_base + st.launch);
            const SlowRange r = {st.lo, st.hi};
            if (rc == DRS_OK) rc = (st.launch & 1) ? launch_one(p, dA, dB, p->hs_run, -1, &r) : launch_one(p, dB, dA, p->hs_run, -1, &r);
            if (rc == DRS_OK && (st.faces & (drs::SIGNAL_LOWER | drs::SIGNAL_UPPER)))
                rc = launch_signal(p, p->hs_run, (st.faces & drs::SIGNAL_LOWER) ? p->lower_flag : nullptr,
                                   (st.faces & drs::SIGNAL_UPPER) ? p->upper_flag : nullptr, flag_base + st.launch + 1);
        } else {
            cudaEventRecord(done[st.block], p->hs_run);
            cudaStreamWaitEvent(p->hs_dn, done[st.block], 0);
            if (st.hi > st.lo)
                cudaMemcpyAsync(host + (st.lo - h0) * unit, dA + st.lo * unit, (size_t)(st.hi - st.lo) * unit, cudaMemcpyDeviceToHost, p->hs_dn);
        }
    }
    cudaEventRecord(fin, p->hs_dn);
    cudaStreamWaitEvent(0, fin, 0);
    cudaEventRecord(e1, 0);
    int rc2 = drs_plan_sync_check(p, nullptr);
    for (cudaStream_t st : {p->hs_up, p->hs_run, p->hs_dn}) cudaStreamSynchronize(st);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(fin);
    for (int b = 0; b < B; ++b) { cudaEventDestroy(up[b]); cudaEventDestroy(done[b]); }
    if (device_ms) *device_ms = ms;
    const cudaError_t ce = cudaGetLastError();
    if (rc == DRS_OK && rc2 == DRS_OK && ce != cudaSuccess) return fail(DRS_E_CUDA, std::string(what) + cudaGetErrorString(ce));
    return rc != DRS_OK ? rc : rc2;
}

// Step list of a streamed drs_run_host; empty when the plain copy-sweep-copy sequence applies.
static std::vector<drs::HostStep> host_steps(const drs_plan* p, int n) {
    const std::vector<int> depth = launch_depths(p, n);
    const long long S = host_block_units(p, depth);
    if (S <= 0) return {};
    return drs::plan_block_schedule(drs::whole_grid(p->local_slow(), p->spec.halo), p->spec.halo, S, depth);
}

// Step list of this rank for a slab host run; empty when the plain sequence applies.
static std::vector<drs::HostStep> slab_steps(const drs_plan* p, int n, bool up_skew) {
    const std::vector<int> depth(n, 1);         // single sweeps: launch_depths is all 1s on slab plans
    const long long S = host_block_units(p, depth, true);
    if (S <= 0) return {};
    const long long H = p->spec.halo, org = p->lo - H;
    drs::SlabSide g;
    g.local = p->local_slow();
    g.own_lo = H; g.own_hi = g.local - H;
    g.out_lo = std::max<long long>(p->lo, H) - org;
    g.out_hi = std::min<long long>(p->hi, p->g_slow - H) - org;
    g.has_lower = p->lo > 0; g.has_upper = p->hi < p->g_slow;
    g.up_skew = up_skew;
    if (g.out_hi - g.out_lo < 2 * H || g.own_hi - g.own_lo <= S) return {};
    return drs::plan_block_schedule(g, H, S, depth);
}

// A step list as records of `width` fields: kind, block, launch, lo, hi (, faces).  Returns the number of steps.
static int step_records(const std::vector<drs::HostStep>& steps, long long* records, int width, int capacity) {
    if (records) {
        if (capacity < (int)steps.size()) return fail(DRS_E_ARG, "buffer too small");
        for (size_t i = 0; i < steps.size(); ++i) {
            const drs::HostStep& st = steps[i];
            long long* r = records + width * i;
            r[0] = st.kind; r[1] = st.block; r[2] = st.launch; r[3] = st.lo; r[4] = st.hi;
            if (width > 5) r[5] = st.faces;
        }
    }
    return (int)steps.size();
}

int drs_plan_host_schedule(const drs_plan* p, int iterations, long long* records5, int capacity) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    return step_records(host_steps(p, sweeps_for(p, iterations)), records5, 5, capacity);
}

int drs_run_host(drs_plan* p, void* h_a, void* h_b, int iterations, float* device_ms) {
    if (!p || !h_a) return fail(DRS_E_ARG, "null argument");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    const size_t bytes = (size_t)p->st.L * p->st.M * p->st.N * p->spec.esize();
    for (int i = 0; i < 2; ++i)
        if (!p->h_dev[i] && cudaMalloc(&p->h_dev[i], bytes) != cudaSuccess)
            return fail(DRS_E_CUDA, "cudaMalloc of the sweep buffers failed");
    const std::vector<drs::HostStep> steps = h_b ? std::vector<drs::HostStep>() : host_steps(p, sweeps_for(p, iterations));
    if (!steps.empty())
        return run_blocks(p, steps, (char*)p->h_dev[0], (char*)p->h_dev[1], (char*)h_a, 0, !p->h_dev_b_ring_zero, 0,
                          "streamed host run: ", device_ms);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, 0);
    cudaMemcpyAsync(p->h_dev[0], h_a, bytes, cudaMemcpyHostToDevice, 0);
    if (h_b) cudaMemcpyAsync(p->h_dev[1], h_b, bytes, cudaMemcpyHostToDevice, 0);
    else cudaMemsetAsync(p->h_dev[1], 0, bytes, 0);   // the reference's h_out is all zeros (getZero2DArray)
    p->h_dev_b_ring_zero = h_b == nullptr;
    rc = run_schedule(p, p->h_dev[0], p->h_dev[1], iterations, nullptr, nullptr, false);
    cudaMemcpyAsync(h_a, p->h_dev[0], bytes, cudaMemcpyDeviceToHost, 0);
    cudaEventRecord(e1, 0);
    int rc2 = drs_plan_sync_check(p, nullptr);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (device_ms) *device_ms = ms;
    return rc != DRS_OK ? rc : rc2;
}

int drs_plan_slab_schedule(const drs_plan* p, int iterations, int up_skew, long long* records6, int capacity) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    if (!p->slab) return fail(DRS_E_ARG, "call drs_plan_set_slab first");
    if (p->slab_pairs) return fail(DRS_E_ARG, "a pair slab (deep ghost planes) has no streamed host schedule");
    return step_records(slab_steps(p, sweeps_for(p, iterations), up_skew != 0), records6, 6, capacity);
}

int drs_plan_set_graph(drs_plan* p, int enable) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    p->use_graph = enable != 0;
    return DRS_OK;
}

int drs_plan_set_host_block(drs_plan* p, long long units) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    p->host_block = units;
    return DRS_OK;
}

int drs_check_error(drs_plan* p, const void* d_out, const void* d_ref, double res[2]) {
    if (!p || !d_out || !d_ref || !res) return fail(DRS_E_ARG, "null argument");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    cudaMemset(p->d_res, 0, 2 * sizeof(double));
    DevParams q;
    fill_params(p, d_out, nullptr, q);
    void* args[] = {&q, (void*)&d_ref, &p->d_res};
    unsigned bx = 32, by = 8;
    unsigned gx = (unsigned)((q.N + bx - 1) / bx), gy = (unsigned)((q.M + by - 1) / by), gz = (unsigned)q.L;
    CUresult r = driver().LaunchKernel(p->f_check, gx, gy, gz, bx, by, 1, 0, nullptr, args, nullptr);
    if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "launch check_: " + cu_err(r));
    p->launches++;
    double h[2];
    if (cudaMemcpy(h, p->d_res, sizeof h, cudaMemcpyDeviceToHost) != cudaSuccess) return fail(DRS_E_CUDA, "result read failed");
    const double cnt = (double)std::max<long long>(1, q.N - 2 * q.halo) * (double)std::max<long long>(1, q.slow_hi - q.slow_lo) *
                       (p->spec.dim == 3 ? (double)std::max<long long>(1, q.M - 2 * q.halo) : 1.0);
    double mx;
    std::memcpy(&mx, &h[0], sizeof mx);
    res[0] = mx > 1e-13 ? mx : 1e-13;   // common.hpp:53 starts the running maximum at 1e-13
    res[1] = std::sqrt(h[1] / cnt);
    return DRS_OK;
}

long long drs_plan_launch_count(const drs_plan* p) { return p ? p->launches : 0; }

// ---- slabs -------------------------------------------------------------------------------
int drs_plan_set_slab(drs_plan* p, long long global_slow, long long lo, long long hi) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    const long long ghost = p->spec.halo;
    if (lo < 0 || hi <= lo || hi > global_slow) return fail(DRS_E_ARG, "bad slab range");
    if (p->spec.sub_launches > 1)
        return fail(DRS_E_ARG, "slab runs cannot use per-sub-step launches: use the fused temporal kernel or --fuse algebraic");
    if (hi - lo + 2 * ghost != p->local_slow())
        return fail(DRS_E_ARG, "slab arrays must hold hi - lo + 2*Halo planes along the slow axis");
    if (drs::has_slab2d_unit(p->spec) && p->slab_cubin.empty()) {
        std::string src = drs::generate_tu(p->spec, true), key;
        std::vector<char> cubin;
        const int rc = compile_cubin(src, cubin, key, Unit::SLAB2D);
        if (rc != DRS_OK) return rc;
        p->slab_source = std::move(src); p->slab_key = std::move(key); p->slab_cubin = std::move(cubin);
    }
    p->slab = true; p->slab_pairs = false; p->g_slow = global_slow; p->lo = lo; p->hi = hi;
    drop_graphs(p);      // launch parameters changed
    return DRS_OK;
}

int drs_plan_set_slab_pairs(drs_plan* p, long long global_slow, long long lo, long long hi) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    const drs::KernelSpec& s = p->spec;
    if (p->slab) return fail(DRS_E_ARG, "this plan is already a slab");
    if (s.dim != 3) return fail(DRS_E_ARG, "pair slabs are 3D only");
    if (s.step != 1 || s.ts != 1 || s.sub_launches > 1) return fail(DRS_E_ARG, "pair slabs need a step-1 plan (two single steps per launch)");
    if (s.reuse) return fail(DRS_E_ARG, "--fuse reuse has no fused halo push: use --fuse temporal or algebraic on a slab");
    if (!drs::fused3d_fits(s.e, s.vec(), 2)) return fail(DRS_E_ARG, "the operator's depth-2 tile keeps no useful columns");
    if (!s.tma_ok)
        return fail(DRS_E_ARG, "this plan runs the naive kernel (operator too deep for the TMA ring), which has no fused halo push");
    if (s.flat) return fail(DRS_E_ARG, "the pair kernel needs a 16-byte row pitch (N a multiple of 2 in fp64, 4 in fp32)");
    if (lo < 0 || hi <= lo || hi > global_slow) return fail(DRS_E_ARG, "bad slab range");
    if (hi - lo + 4LL * s.halo != p->local_slow())
        return fail(DRS_E_ARG, "pair slab arrays must hold hi - lo + 4*Halo planes along the slow axis");
    drs::KernelSpec ps;
    if (!drs::pair_spec(p->st, s, ps, false)) return fail(DRS_E_ARG, "no pair kernel for this operator's tile");
    std::string src = drs::generate_slabpair_tu(ps), key;
    std::vector<char> cubin;
    const int rc = compile_cubin(src, cubin, key, Unit::SLABPAIR);
    if (rc != DRS_OK) return rc;
    p->pspec = ps;       // the same specialisation as drs_run's pair unit where the plan has one
    p->ptmaps.clear();
    p->slabpair_source = std::move(src); p->slabpair_key = std::move(key); p->slabpair_cubin = std::move(cubin);
    p->slab = true; p->slab_pairs = true; p->g_slow = global_slow; p->lo = lo; p->hi = hi;
    drop_graphs(p);
    return p->loaded ? load_slabpair(p) : DRS_OK;
}

int drs_plan_slab_split(const drs_plan* p, int iterations, int* pairs, int* singles) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    const int n = sweeps_for(p, iterations);
    int np = 0, ns = n;
    if (p->slab_pairs) drs::pair_split(n, np, ns);
    if (pairs) *pairs = np;
    if (singles) *singles = ns;
    return n;
}

int drs_sweep_pair(drs_plan* p, const void* d_in, void* d_out, void* stream) {
    if (!p || !d_in || !d_out) return fail(DRS_E_ARG, "null argument");
    if (!p->slab_pairs || !p->my_bases[0] || !p->my_bases[1])
        return fail(DRS_E_ARG, "call drs_plan_set_slab_pairs and drs_plan_set_peers first");
    if (!((d_in == p->my_bases[0] && d_out == p->my_bases[1]) || (d_in == p->my_bases[1] && d_out == p->my_bases[0])))
        return fail(DRS_E_ARG, "a pair launch runs between the two arrays given to drs_plan_set_peers");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    return launch_slabpair(p, d_in, d_out, (cudaStream_t)stream, -1);
}

int drs_plan_set_peers(drs_plan* p, void* const my_bases[2], void* const lower_bases[2], void* const upper_bases[2],
                       long long lower_lo, long long upper_lo) {
    if (!p || !my_bases) return fail(DRS_E_ARG, "null argument");
    if (!p->slab) return fail(DRS_E_ARG, "call drs_plan_set_slab first");
    if (p->spec.reuse) return fail(DRS_E_ARG, "--fuse reuse has no fused halo push: use --fuse temporal or algebraic on a slab");
    if (!p->spec.tma_ok)
        return fail(DRS_E_ARG, "this plan runs the naive kernel (operator too deep for the TMA ring), which has no fused halo push");
    for (int b = 0; b < 2; ++b)
        for (const void* q : {(const void*)my_bases[b], lower_bases ? (const void*)lower_bases[b] : nullptr,
                              upper_bases ? (const void*)upper_bases[b] : nullptr})
            if ((reinterpret_cast<uintptr_t>(q) & 15) != 0) return fail(DRS_E_ARG, "slab array bases must be 16-byte aligned");
    for (int b = 0; b < 2; ++b) {
        p->my_bases[b] = my_bases[b];
        p->lower_bases[b] = lower_bases ? lower_bases[b] : nullptr;
        p->upper_bases[b] = upper_bases ? upper_bases[b] : nullptr;
    }
    p->lower_lo = lower_lo; p->upper_lo = upper_lo;
    drop_graphs(p);      // launch parameters changed
    return DRS_OK;
}

int drs_signal_peers(drs_plan* p, void* lower_flag, void* upper_flag, long long value, void* stream) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    return launch_signal(p, (cudaStream_t)stream, lower_flag, upper_flag, value);
}

int drs_wait_flags(drs_plan* p, const void* my_flags, int wait_lower, int wait_upper, long long value, void* stream) {
    if (!p || !my_flags) return fail(DRS_E_ARG, "null argument");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    return launch_wait(p, (cudaStream_t)stream, my_flags, wait_lower, wait_upper, value);
}

int drs_plan_set_flags(drs_plan* p, const void* my_flags, void* lower_flag, void* upper_flag) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    if (!p->slab || !p->my_bases[0] || !p->my_bases[1]) return fail(DRS_E_ARG, "call drs_plan_set_slab and drs_plan_set_peers first");
    if (!my_flags) return fail(DRS_E_ARG, "my_flags is null");
    for (const void* q : {my_flags, (const void*)lower_flag, (const void*)upper_flag})
        if ((reinterpret_cast<uintptr_t>(q) & 7) != 0) return fail(DRS_E_ARG, "flag words must be 8-byte aligned");
    p->my_flags = my_flags; p->lower_flag = lower_flag; p->upper_flag = upper_flag;
    drop_graphs(p);
    return DRS_OK;
}

// One rank's share of the emitted host loop on a slab-decomposed grid.  One launch per sweep: the sweep
// kernel waits for / signals its neighbours itself (Params::my_flags ...), the launches are replayed as a
// CUDA graph, and the only thing that changes between calls -- the flag value of the call's first sweep --
// lives in device memory and is written in stream order before the replay.
int drs_run_slab(drs_plan* p, int iterations, void* stream_, int* sweeps) {
    if (!p) return fail(DRS_E_ARG, "null plan");
    if (!p->slab || !p->my_bases[0] || !p->my_bases[1]) return fail(DRS_E_ARG, "call drs_plan_set_slab and drs_plan_set_peers first");
    const bool alone = !p->lower_bases[0] && !p->upper_bases[0];
    if (!alone && !p->my_flags) return fail(DRS_E_ARG, "call drs_plan_set_flags first");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!p->d_sync) {
        if (cudaMalloc(&p->d_sync, 16) != cudaSuccess) return fail(DRS_E_CUDA, "cudaMalloc(slab sync words)");
        cudaMemset(p->d_sync, 0, 16);
    }
    const int n = sweeps_for(p, iterations);
    if (sweeps) *sweeps = n;
    if (n == 0) return DRS_OK;
    // pair slabs: `pairs` pair launches, then `singles` single sweeps; flag values count launches
    int pairs = 0, singles = n;
    if (p->slab_pairs) drs::pair_split(n, pairs, singles);
    // flag value of this call's launch 0, in stream order (no kernel)
    const long long base = p->slab_seq;
    if (driver().StreamWriteValue64) {
        CUresult r = driver().StreamWriteValue64((CUstream)stream, (CUdeviceptr)p->d_sync, (cuuint64_t)base, 0);
        if (r != CUDA_SUCCESS) return fail(DRS_E_CUDA, "cuStreamWriteValue64: " + cu_err(r));
    } else if (cudaMemcpyAsync(p->d_sync, &base, sizeof base, cudaMemcpyHostToDevice, stream) != cudaSuccess) {
        return fail(DRS_E_CUDA, "slab sequence base upload failed");      // pageable source: staged before return
    }
    void* a = p->my_bases[0];
    void* b = p->my_bases[1];
    auto enqueue = [&](cudaStream_t st) -> int {
        int r = DRS_OK;
        for (int i = 0; i < pairs && r == DRS_OK; ++i)
            r = (i & 1) ? launch_slabpair(p, b, a, st, i) : launch_slabpair(p, a, b, st, i);
        for (int s = 0; s < singles && r == DRS_OK; ++s)
            r = (s & 1) ? launch_one(p, b, a, st, -1, nullptr, pairs + s) : launch_one(p, a, b, st, -1, nullptr, pairs + s);
        return r;
    };
    if (!run_graph(p, a, b, n, true, stream, enqueue) && (rc = enqueue(stream)) != DRS_OK) return rc;
    p->slab_seq += pairs + singles;
    return DRS_OK;
}

// Executor of drs_plan_slab_schedule (validated on 2, 4 and 8 GPUs: bit-exact against the single-GPU run,
// tools/slab_check.py and bench.py's in-run parity): one rank's share of a slab-decomposed host-buffer run, on
// the block executor of drs_run_host.  h_own holds the rank's own planes, local planes [H, local - H).  Flags are
// monotone: this call uses the values slab_seq + 1 ... slab_seq + sweeps + 1 and leaves slab_seq at the largest
// one; the caller separates calls by a barrier.
int drs_run_host_slab(drs_plan* p, void* h_own, int iterations, int up_skew, float* device_ms) {
    if (!p || !h_own) return fail(DRS_E_ARG, "null argument");
    if (!p->slab || !p->my_bases[0] || !p->my_bases[1]) return fail(DRS_E_ARG, "call drs_plan_set_slab and drs_plan_set_peers first");
    if (!p->my_flags) return fail(DRS_E_ARG, "call drs_plan_set_flags first");
    if (p->slab_pairs) return fail(DRS_E_ARG, "a pair slab (deep ghost planes) has no streamed host run");
    int rc = ensure_loaded(p);
    if (rc != DRS_OK) return rc;
    const int n = sweeps_for(p, iterations);
    const std::vector<drs::HostStep> steps = slab_steps(p, n, up_skew != 0);
    if (steps.empty()) return fail(DRS_E_ARG, "no streamed schedule for this slab (too thin, or switched off): use the plain sequence");
    rc = run_blocks(p, steps, (char*)p->my_bases[0], (char*)p->my_bases[1], (char*)h_own, p->spec.halo, false, p->slab_seq,
                    "streamed slab run: ", device_ms);
    if (rc == DRS_OK) p->slab_seq += n + 1;    // the largest flag value this call wrote
    return rc;
}

int drs_ipc_export(void* d_ptr, unsigned char handle[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, d_ptr);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
    std::memcpy(handle, &h, 64);
    return DRS_OK;
}
int drs_ipc_import(const unsigned char handle[64], void** d_ptr) {
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    cudaError_t e = cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
    return DRS_OK;
}
int drs_ipc_close(void* d_ptr) {
    cudaError_t e = cudaIpcCloseMemHandle(d_ptr);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("cudaIpcCloseMemHandle: ") + cudaGetErrorString(e));
    return DRS_OK;
}
int drs_device_malloc(size_t bytes, void** d_ptr) {
    cudaError_t e = cudaMalloc(d_ptr, bytes);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    return DRS_OK;
}
int drs_device_free(void* d_ptr) { cudaFree(d_ptr); return DRS_OK; }
int drs_device_upload(void* d_dst, const void* h_src, size_t bytes) {
    cudaError_t e = cudaMemcpy(d_dst, h_src, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("cudaMemcpy H2D: ") + cudaGetErrorString(e));
    return DRS_OK;
}
int drs_device_download(void* h_dst, const void* d_src, size_t bytes) {
    cudaError_t e = cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("cudaMemcpy D2H: ") + cudaGetErrorString(e));
    return DRS_OK;
}

// ---- emitters ----------------------------------------------------------------------------
int drs_emit_program(const drs_stencil* s, const drs_knobs* k, const char* kernel_name, const char* path) {
    if (!s || !k || !path) return fail(DRS_E_ARG, "null argument");
    drs::KernelSpec spec;
    spec.name = kernel_name && *kernel_name ? kernel_name : s->name;
    std::string err = drs::choose_spec(s->st, *k, spec);
    if (!err.empty()) return fail(DRS_E_ARG, err);
    std::ofstream f(path, std::ios::out | std::ios::trunc);
    if (!f) return fail(DRS_E_IO, std::string("cannot write ") + path);
    f << drs::emit_program_text(s->st, *k, spec);
    return DRS_OK;
}

const char* drs_last_error(void) { return g_err.c_str(); }
const char* drs_version(void) { return "drstencil-b200 0.2 (sm_100a)"; }
const char* drs_compiler(void) {
    static std::string text;
    Nvrtc& n = nvrtc();
    int maj = 0, min = 0;
    if (n.ok) n.Version(&maj, &min);
    text = n.ok ? "NVRTC " + std::to_string(maj) + "." + std::to_string(min) + " (" + n.path + ")" : "NVRTC unavailable: " + n.why;
    return text.c_str();
}
int drs_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int drs_set_device(int ordinal) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return fail(DRS_E_NOGPU, "drstencil needs a CUDA device (no CPU fallback)"); }
    if (ordinal < 0 || ordinal >= n) return fail(DRS_E_ARG, "no CUDA device " + std::to_string(ordinal));
    cudaError_t e = cudaSetDevice(ordinal);
    if (e != cudaSuccess) return fail(DRS_E_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    return DRS_OK;
}
void drs_set_cache_dir(const char* dir) { g_cache_dir = dir ? dir : ""; }

}  // extern "C"
