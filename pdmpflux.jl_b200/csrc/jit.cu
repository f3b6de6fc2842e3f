// Source potentials: user-written CUDA (jit_source.cuh states the contract) compiled at run time with NVRTC into the
// thinning kernels of chain.cuh -- the generic one, or the fast paths for a source that declares a line model -- then
// loaded and launched like the built-in instantiations.
//
// NVRTC is bound at run time (dlopen), so the library keeps no link-time dependency on it.  The toolkit the library was
// built with is tried first: the process may already hold another libnvrtc.so.12 (PyTorch bundles one), and a
// different compiler version would not reproduce the built-in kernels bit for bit.  The headers the kernels need are
// compiled into the library as strings (generated from the files themselves by the Makefile), so running needs
// nothing but libnvrtc.
//
// Compiled cubins live in one process-wide cache keyed by everything that determines them (source, headers, NVRTC
// version, sampler kind, team width, path, line model, defines) -- not by the potential handle, which the Python binding creates afresh
// for every sampler.  Parameters are run-time data and never part of the key.
#include <dlfcn.h>

#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <type_traits>

#include "common.cuh"
#include "jit.cuh"

int pdmpflux_fail_(int code, const std::string& msg);  // api.cu: sets the thread-local error message

#ifndef PDMPFLUX_CUDA_HOME
#define PDMPFLUX_CUDA_HOME "/usr/local/cuda"
#endif
#define PDMPFLUX_STR2(x) #x
#define PDMPFLUX_STR(x) PDMPFLUX_STR2(x)

namespace pdmpflux {
namespace {

struct EmbeddedHeader { const char* name; const char* text; };
const EmbeddedHeader kHeaders[] = {
#include "jit_headers.inc"
};
constexpr int kNumHeaders = sizeof(kHeaders) / sizeof(kHeaders[0]);
constexpr size_t kMaxLog = 16 * 1024;   // bytes of NVRTC log kept in the error message

// ---- NVRTC, bound at run time ----------------------------------------------------------------------------
struct Nvrtc {
    using Prog = void*;
    void* lib = nullptr;
    int (*Version)(int*, int*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    int (*CreateProgram)(Prog*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*DestroyProgram)(Prog*) = nullptr;
    int (*AddNameExpression)(Prog, const char*) = nullptr;
    int (*CompileProgram)(Prog, int, const char* const*) = nullptr;
    int (*GetProgramLogSize)(Prog, size_t*) = nullptr;
    int (*GetProgramLog)(Prog, char*) = nullptr;
    int (*GetCUBINSize)(Prog, size_t*) = nullptr;
    int (*GetCUBIN)(Prog, char*) = nullptr;
    int (*GetLoweredName)(Prog, const char*, const char**) = nullptr;
    std::string version, why;
};

Nvrtc& nvrtc() {
    static Nvrtc n;
    static std::once_flag once;
    std::call_once(once, [] {
        const std::string soname = "libnvrtc.so." PDMPFLUX_STR(__CUDACC_VER_MAJOR__);
        const std::string names[] = {std::string(PDMPFLUX_CUDA_HOME) + "/lib64/" + soname, soname, "libnvrtc.so"};
        for (const std::string& nm : names)
            if ((n.lib = dlopen(nm.c_str(), RTLD_NOW | RTLD_LOCAL))) break;
        if (!n.lib) { n.why = "NVRTC (" + soname + ") not found: source potentials need the CUDA run-time compiler"; return; }
        bool ok = true;
        auto sym = [&](auto& fn, const char* name) {
            fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(n.lib, name));
            ok = ok && fn != nullptr;
        };
        sym(n.Version, "nvrtcVersion"); sym(n.GetErrorString, "nvrtcGetErrorString");
        sym(n.CreateProgram, "nvrtcCreateProgram"); sym(n.DestroyProgram, "nvrtcDestroyProgram");
        sym(n.AddNameExpression, "nvrtcAddNameExpression"); sym(n.CompileProgram, "nvrtcCompileProgram");
        sym(n.GetProgramLogSize, "nvrtcGetProgramLogSize"); sym(n.GetProgramLog, "nvrtcGetProgramLog");
        sym(n.GetCUBINSize, "nvrtcGetCUBINSize"); sym(n.GetCUBIN, "nvrtcGetCUBIN");
        sym(n.GetLoweredName, "nvrtcGetLoweredName");
        int major = 0, minor = 0;
        if (!ok || n.Version(&major, &minor) != 0) {
            dlclose(n.lib);
            n.lib = nullptr;
            n.why = "the NVRTC library found lacks the entry points source potentials need";
            return;
        }
        n.version = std::to_string(major) + "." + std::to_string(minor);
    });
    return n;
}

// the host's KernelParams size: jit_source.cuh checks that the run-time kernels see the same layout
std::string defines() {
    return "#define PDMPFLUX_HOST_KERNEL_PARAMS_BYTES " + std::to_string(sizeof(KernelParams)) + "\n";
}

struct Entry {
    std::string cubin, lowered;
    SourceTraits traits;               // the contract check: what the source declares
    cudaLibrary_t library = nullptr;   // loaded on first launch (context independent: serves every device)
    cudaKernel_t kernel = nullptr;
};

struct Cache {
    std::mutex mu;
    std::map<std::string, std::unique_ptr<Entry>> entries;
    std::atomic<int64_t> compiles{0};
};
Cache& cache() {
    static Cache* c = new Cache();   // never destroyed: loaded libraries must outlive static destruction order
    return *c;
}

uint64_t fnv1a(const std::string& s, uint64_t h = 1469598103934665603ull) {
    for (unsigned char ch : s) { h ^= ch; h *= 1099511628211ull; }
    return h;
}
uint64_t headers_hash() {
    static const uint64_t h = [] {
        uint64_t x = 1469598103934665603ull;
        for (const EmbeddedHeader& e : kHeaders) x = fnv1a(std::string(e.name) + '\0' + e.text, x);
        return x;
    }();
    return h;
}

// kind < 0: the contract-check program; otherwise the skeleton kernels.  The check also instantiates an empty kernel
// whose template arguments are the traits of Pot<PDMPFLUX_SOURCE>: its lowered (mangled) name carries them back to the
// host without a CUDA call.
const char kTraitsName[] = "&pdmpflux_traits<pdmpflux::Pot<PDMPFLUX_SOURCE>::K, pdmpflux::Pot<PDMPFLUX_SOURCE>::kAffine, "
                           "pdmpflux::Pot<PDMPFLUX_SOURCE>::kSpecial, pdmpflux::Pot<PDMPFLUX_SOURCE>::kSplit>";
std::string program_text(const std::string& source, int kind) {
    std::string s = defines();
    s += "#include \"potentials.cuh\"\n#line 1 \"user_potential\"\n";
    s += source;
    s += "\n#include \"jit_source.cuh\"\n";
    if (kind < 0)
        s += "__global__ void pdmpflux_contract_check(pdmpflux::PotParams pp, double* out) {\n"
             "    using P = pdmpflux::Pot<PDMPFLUX_SOURCE>;\n"
             "    double acc[P::K > 0 ? P::K : 1] = {}, Ld[P::K > 0 ? P::K : 1] = {}, g = 0.0, hd = 0.0;\n"
             "    P::accum(pp, threadIdx.x, out[0], acc);\n"
             "    P::eval(pp, threadIdx.x, out[0], out[1], acc, Ld, g, hd);\n"
             "    out[2] = P::grad(pp, threadIdx.x, out[0], acc) + g + hd;\n"
             "}\n"
             "template <int K, bool Affine, int Special, bool Split> __global__ void pdmpflux_traits() {}\n";
    else s += "#include \"chain.cuh\"\n";
    return s;
}

std::string kernel_name(int kind, int team, int path, int nw) {
    return "pdmpflux::skeleton_kernel<" + std::to_string(team) + ", " + std::to_string(kind) + ", " +
           std::to_string((int)PDMPFLUX_SOURCE) + ", " + std::to_string(path) + ", " + std::to_string(nw) + ">";
}

// Reads the template arguments of pdmpflux_traits<K, kAffine, kSpecial, kSplit> out of its Itanium-mangled name,
// e.g. _Z15pdmpflux_traitsILi2ELb1ELi2ELb0EEvv: integer literals "L<type><value>E", a negative value as "n<digits>".
bool parse_traits(const std::string& lowered, SourceTraits& t) {
    const size_t open = lowered.find("pdmpflux_traitsI");
    if (open == std::string::npos) return false;
    size_t pos = open + sizeof("pdmpflux_traitsI") - 1;
    const char types[4] = {'i', 'b', 'i', 'b'};
    long v[4];
    for (int k = 0; k < 4; ++k) {
        if (pos + 2 >= lowered.size() || lowered[pos] != 'L' || lowered[pos + 1] != types[k]) return false;
        pos += 2;
        const bool neg = lowered[pos] == 'n';
        if (neg) ++pos;
        size_t digits = 0;
        long x = 0;
        while (pos < lowered.size() && lowered[pos] >= '0' && lowered[pos] <= '9' && digits < 9) {
            x = 10 * x + (lowered[pos++] - '0');
            ++digits;
        }
        if (digits == 0 || pos >= lowered.size() || lowered[pos++] != 'E') return false;
        v[k] = neg ? -x : x;
    }
    if (pos >= lowered.size() || lowered[pos] != 'E') return false;
    t.K = (int)v[0]; t.affine = v[1] != 0; t.special = (int)v[2]; t.split = v[3] != 0;
    return true;
}

// Compiles (or finds) the program for (source, kind, team, path, nw).  Caller holds the cache mutex.
int get_entry(const std::string& source, int kind, int team, int path, int nw, Entry** out) {
    Nvrtc& nv = nvrtc();
    if (!nv.lib) return pdmpflux_fail_(PDMPFLUX_ERR_UNSUPPORTED, nv.why);
    const std::string text = program_text(source, kind);
    const std::string key = nv.version + '\0' + std::to_string(headers_hash()) + '\0' + std::to_string(kind) + '\0' +
                            std::to_string(team) + '\0' + std::to_string(path) + '\0' + std::to_string(nw) + '\0' + text;
    Cache& c = cache();
    auto it = c.entries.find(key);
    if (it != c.entries.end()) { *out = it->second.get(); return PDMPFLUX_OK; }

    const char* names[kNumHeaders];
    const char* texts[kNumHeaders];
    for (int i = 0; i < kNumHeaders; ++i) { names[i] = kHeaders[i].name; texts[i] = kHeaders[i].text; }
    Nvrtc::Prog prog = nullptr;
    int r = nv.CreateProgram(&prog, text.c_str(), "pdmpflux_source_potential.cu", kNumHeaders, texts, names);
    if (r != 0) return pdmpflux_fail_(PDMPFLUX_ERR_COMPILE, std::string("nvrtcCreateProgram: ") + nv.GetErrorString(r));
    struct Guard { Nvrtc& nv; Nvrtc::Prog* p; ~Guard() { nv.DestroyProgram(p); } } guard{nv, &prog};
    const std::string name = kind < 0 ? std::string(kTraitsName) : kernel_name(kind, team, path, nw);
    if ((r = nv.AddNameExpression(prog, name.c_str())) != 0)
        return pdmpflux_fail_(PDMPFLUX_ERR_COMPILE, std::string("nvrtcAddNameExpression: ") + nv.GetErrorString(r));
    // nvcc's defaults (what the built-in kernels are compiled with), stated explicitly
    const char* opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "--fmad=true", "--ftz=false", "--prec-div=true",
                          "--prec-sqrt=true"};
    r = nv.CompileProgram(prog, (int)(sizeof(opts) / sizeof(opts[0])), opts);
    c.compiles.fetch_add(1);
    if (r != 0) {
        size_t n = 0;
        std::string log;
        if (nv.GetProgramLogSize(prog, &n) == 0 && n > 1) {
            log.resize(n);
            nv.GetProgramLog(prog, &log[0]);
            log.resize(n - 1);
        }
        if (log.size() > kMaxLog) log = log.substr(0, kMaxLog) + "\n... (log truncated)";
        return pdmpflux_fail_(PDMPFLUX_ERR_COMPILE, "source potential failed to compile (NVRTC " + nv.version + ", " +
                                                        (kind < 0 ? std::string("contract check") : name) + "):\n" + log);
    }
    auto e = std::make_unique<Entry>();
    if (kind < 0) {
        const char* lowered = nullptr;
        if (nv.GetLoweredName(prog, name.c_str(), &lowered) != 0 || !lowered || !parse_traits(lowered, e->traits))
            return pdmpflux_fail_(PDMPFLUX_ERR_COMPILE, "NVRTC " + nv.version + ": cannot read the potential's traits from the "
                                                        "lowered name '" + std::string(lowered ? lowered : "(none)") + "'");
    } else {
        size_t n = 0;
        const char* lowered = nullptr;
        if (nv.GetCUBINSize(prog, &n) != 0 || n == 0 || nv.GetLoweredName(prog, name.c_str(), &lowered) != 0 || !lowered)
            return pdmpflux_fail_(PDMPFLUX_ERR_COMPILE, "NVRTC " + nv.version + " produced no cubin for " + name);
        e->cubin.resize(n);
        nv.GetCUBIN(prog, &e->cubin[0]);
        e->lowered = lowered;
    }
    *out = e.get();
    c.entries.emplace(key, std::move(e));
    return PDMPFLUX_OK;
}

}  // namespace

int jit_check_source(const std::string& source, SourceTraits* traits) {
    std::lock_guard<std::mutex> lk(cache().mu);
    Entry* e = nullptr;
    const int rc = get_entry(source, -1, 0, kPathGeneric, kLineShared, &e);
    if (rc == PDMPFLUX_OK && traits) *traits = e->traits;
    return rc;
}

int jit_prepare(const std::string& source, int sampler_kind, int team, int path, int nw) {
    std::lock_guard<std::mutex> lk(cache().mu);
    Entry* e = nullptr;
    return get_entry(source, sampler_kind, team, path, nw, &e);
}

int jit_launch(const std::string& source, int sampler_kind, int team, int path, int nw, const KernelParams& p,
               unsigned grid, size_t smem, cudaStream_t stream) {
    Entry* e = nullptr;
    {
        std::lock_guard<std::mutex> lk(cache().mu);
        int rc = get_entry(source, sampler_kind, team, path, nw, &e);
        if (rc != PDMPFLUX_OK) return rc;
        if (!e->kernel) {
            cudaError_t ce = cudaLibraryLoadData(&e->library, e->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
            if (ce == cudaSuccess) ce = cudaLibraryGetKernel(&e->kernel, e->library, e->lowered.c_str());
            if (ce != cudaSuccess) {
                e->kernel = nullptr;
                return pdmpflux_fail_(PDMPFLUX_ERR_CUDA, std::string("loading the source-potential kernel: ") + cudaGetErrorString(ce));
            }
        }
    }
    if (smem > 48 * 1024) {
        int dev = 0;
        cudaError_t ce = cudaGetDevice(&dev);
        if (ce == cudaSuccess) ce = cudaKernelSetAttributeForDevice(e->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem, dev);
        if (ce != cudaSuccess) return pdmpflux_fail_(PDMPFLUX_ERR_CUDA, std::string("source-potential kernel attribute: ") + cudaGetErrorString(ce));
    }
    void* args[] = {const_cast<KernelParams*>(&p)};
    const cudaError_t ce = cudaLaunchKernel(reinterpret_cast<const void*>(e->kernel), dim3(grid),
                                            dim3(block_threads_rt(team, sampler_kind, path, PDMPFLUX_SOURCE)), args, smem, stream);
    if (ce != cudaSuccess) return pdmpflux_fail_(PDMPFLUX_ERR_CUDA, std::string("skeleton kernel launch (source potential): ") + cudaGetErrorString(ce));
    return PDMPFLUX_OK;
}

int64_t jit_compile_count() { return cache().compiles.load(); }

}  // namespace pdmpflux
