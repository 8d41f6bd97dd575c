// sp_engine.cu — host side of the C ABI declared in include/spectro_b200.h.
//
// Re-hosts what the reference worker does around its hot loops (lib/worker.js:23-62,
// 140-155): argument unpacking, derived constants, output allocation, and the reply.
// No CPU fallback exists: without an sm_100 device sp_create fails with SP_E_NO_DEVICE.
#include "../../include/spectro_b200.h"
#include "sp_aux_kernels.cuh"
#include "sp_inst.cuh"

#include <cmath>
#include <dlfcn.h>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <strings.h>
#include <thread>
#include <vector>

using sp::Params;

// ---- per-format kernels: sp_inst_<tag>.cu exports sp_kernels_<tag> (weak: a build may carry any subset, "rt" is mandatory)
#define SP_DECL(tag) extern "C" const sp::Kernels sp_kernels_##tag __attribute__((weak));
SP_DECL(rt) SP_DECL(cu4) SP_DECL(cs4) SP_DECL(cu8) SP_DECL(cs8) SP_DECL(cu12) SP_DECL(cs12) SP_DECL(cu16)
SP_DECL(cs16) SP_DECL(cu32) SP_DECL(cs32) SP_DECL(cu64) SP_DECL(cs64) SP_DECL(cf32) SP_DECL(cf64)

// the format's own build, null when the library carries none
static const sp::Kernels *own_kernels(int fmt)
{
    static const sp::Kernels *const tab[SP_FORMAT_COUNT] = { &sp_kernels_cu4, &sp_kernels_cs4, &sp_kernels_cu8, &sp_kernels_cs8,
        &sp_kernels_cu12, &sp_kernels_cs12, &sp_kernels_cu16, &sp_kernels_cs16, &sp_kernels_cu32, &sp_kernels_cs32,
        &sp_kernels_cu64, &sp_kernels_cs64, &sp_kernels_cf32, &sp_kernels_cf64 };
    return tab[fmt];
}
static bool specialised(int fmt) { return own_kernels(fmt) != nullptr; }
// The launchers of format fmt: its own build, else the runtime-switch build's render, prepass and big.  r64, rc and w stage raw
// frames of one sample format and exist for specialised formats only.
static const sp::Kernels &kernels_for(int fmt)
{
    static const sp::Kernels rt = &sp_kernels_rt ? sp::Kernels{ sp_kernels_rt.render, sp_kernels_rt.prepass, nullptr, nullptr, nullptr, sp_kernels_rt.big }
                                                  : sp::Kernels{};
    const sp::Kernels *own = own_kernels(fmt);
    return own ? *own : rt;
}

// ------------------------------------------------------------------ formats (lib/samples.js:22-155)
static const char *const k_names[SP_FORMAT_COUNT] = { "CU4", "CS4", "CU8", "CS8", "CU12", "CS12", "CU16", "CS16",
                                                       "CU32", "CS32", "CU64", "CS64", "CF32", "CF64" };

extern "C" int sp_abi_version(void) { return SP_ABI_VERSION; }
#ifndef SP_BUILD_ID
#define SP_BUILD_ID "unknown"
#endif
extern "C" const char *sp_build_id(void) { return SP_BUILD_ID; }

extern "C" int sp_format_from_name(const char *name)
{
    if (!name) return SP_CU8;
    for (int i = 0; i < SP_FORMAT_COUNT; i++)
        if (!strcasecmp(name, k_names[i])) return i;
    if (!strcasecmp(name, "DATA") || !strcasecmp(name, "COMPLEX16U")) return SP_CU8;
    if (!strcasecmp(name, "COMPLEX16S")) return SP_CS8;
    if (!strcasecmp(name, "CFILE") || !strcasecmp(name, "COMPLEX")) return SP_CF32;
    return SP_CU8;   // lib/samples.js:149-155: anything else is treated as CU8
}
extern "C" const char *sp_format_name(int f) { return (f < 0 || f >= SP_FORMAT_COUNT) ? "?" : k_names[f]; }
extern "C" int sp_sample_width(int f) { return (f < 0 || f >= SP_FORMAT_COUNT) ? SP_E_BAD_FORMAT : sp::sample_width(f); }
extern "C" int sp_element_size(int f) { return (f < 0 || f >= SP_FORMAT_COUNT) ? SP_E_BAD_FORMAT : sp::element_size(f); }

// ------------------------------------------------------------------ NCCL, loaded at run time
// Only a multi-device engine needs it (the merge of lib/spectroplot.js:1229-1238 across GPUs), so the library is opened with
// dlopen when such an engine is created: a single-GPU host needs no NCCL installation, and the .so keeps linking the CUDA
// runtime only.  The handful of types below are NCCL's stable C ABI (nccl.h).
typedef struct ncclComm *sp_ncclComm_t;
enum { SP_NCCL_UINT64 = 5, SP_NCCL_FLOAT64 = 8, SP_NCCL_SUM = 0, SP_NCCL_MAX = 2, SP_NCCL_MIN = 3 };
struct NcclApi {
    void *lib = nullptr;
    int (*CommInitAll)(sp_ncclComm_t *, int, const int *) = nullptr;
    int (*CommDestroy)(sp_ncclComm_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, sp_ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    std::string err;
};
static NcclApi *nccl_api()
{
    static NcclApi api;
    static bool tried = false;
    if (tried) return &api;
    tried = true;
    const char *names[] = { getenv("SP_NCCL_LIB"), "libnccl.so.2", "libnccl.so" };
    for (const char *nm : names) {
        if (!nm || !*nm) continue;
        api.lib = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
        if (api.lib) break;
    }
    if (!api.lib) { api.err = std::string("dlopen(libnccl.so.2): ") + (dlerror() ? dlerror() : "not found"); return &api; }
    auto sym = [&](const char *s) { void *f = dlsym(api.lib, s); if (!f && api.err.empty()) api.err = std::string("missing symbol ") + s; return f; };
    api.CommInitAll = (int (*)(sp_ncclComm_t *, int, const int *))sym("ncclCommInitAll");
    api.CommDestroy = (int (*)(sp_ncclComm_t))sym("ncclCommDestroy");
    api.AllReduce = (int (*)(const void *, void *, size_t, int, int, sp_ncclComm_t, cudaStream_t))sym("ncclAllReduce");
    api.GroupStart = (int (*)())sym("ncclGroupStart");
    api.GroupEnd = (int (*)())sym("ncclGroupEnd");
    api.GetErrorString = (const char *(*)(int))sym("ncclGetErrorString");
    if (!api.err.empty()) { dlclose(api.lib); api.lib = nullptr; }
    return &api;
}

// ------------------------------------------------------------------ engine state
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

// where a shard's image goes inside the caller's [n][total width] picture (multi-device engines; spectrogram layout)
struct Placement { long long pitch_frames; long long col0; };

// kinds of twiddle table (get_table)
enum class Tw { big, passA, passB, tw14, w };

struct sp_engine {
    std::vector<sp_engine *> subs;           // ndev > 1: one single-device engine per GPU; this object only dispatches
    std::vector<sp_ncclComm_t> comms;        // ndev > 1: one NCCL communicator per device (ncclCommInitAll), empty when NCCL is unavailable
    std::string nccl_err;                    // why `comms` is empty
    int cur = 0;                             // sub-engine addressed by the memory helpers / taps (sp_select_device)
    int ndev = 1;
    int dev = 0;
    int sm_count = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    std::string plan;
    std::map<std::pair<Tw, int>, float2 *> tw;   // twiddle tables by (kind, n)
    DevBuf pin[2], pimg[2];                  // pipeline: double-buffered input bytes / image tiles
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_in[2] = { nullptr, nullptr }, ev_comp[2] = { nullptr, nullptr }, ev_out[2] = { nullptr, nullptr }, ev_setup = nullptr;
    DevBuf acc, jhtab;                       // self-cleaning 64-bit histogram accumulators [1000 + SP_MAX_CMAP]; decode table of the joint histogram
    float jhtab_key[5] = { 0, 0, 0, 0, -1 };  // constants the table was built for (jA, jB, jC, jD, cmap_len)
    bool acc_dirty = true;                   // a render was abandoned half way (or nothing is initialised yet): reset the accumulators first
    DevBuf ring, ringctl;                    // n > 4096: L2-resident pre-pass ring and its queue / hand-off counters
    size_t l2_window = 0;                    // bytes of the ring currently covered by the persisting access-policy window
    DevBuf in, zin, spec, image, fmin, fmax, fmid, gauges, hist, jhist, stats, mm, lut, window, window_t, scratch, db, synth_lut;
    // state of an enqueued (not yet finished) render
    std::vector<cudaEvent_t> prof0, prof1;   // per-launch timing ring of the render kernel
    long long prof_count = 0, prof_seq = 0;
    int prof_every = 1;
    bool prof_this = false;
    std::vector<float> h_window, h_window_t; // last uploaded window / LUT (upload only on change)
    std::vector<uint32_t> h_lut;
    double *stats_src = nullptr;             // dBfs min / max of the last prepared render (set by prepare)
    // sp_render_async: up to two host-buffer messages in flight (the copy-out tail of one overlaps the copy-in head of the next)
    struct Inflight {
        cudaEvent_t done = nullptr, reply = nullptr;
        uint8_t *bounce = nullptr;           // pinned: stats and the five small reply arrays (layout: Bounce)
        size_t bounce_cap = 0;
        sp_reply *rp = nullptr;
        long long width = 0;
        int cmap_len = 0, launches = 0, ticket = -1;
        bool busy = false;
    } inflight[2];
    int next_ticket = 0;
    cudaStream_t s_done = nullptr;
    bool pipe_used[2] = { false, false };    // pin[b] / pimg[b] have been used by an earlier chunk (of this or of the previous message)
    bool ev_out_valid[2] = { false, false }; // ev_out[b] has been recorded
    bool pending = false;
    long long pend_width = 0;
    int pend_cmap_len = 0;
    int launches = 0;
    // render_r64_kernel / finalize_kernel overlap (programmatic dependent launch, see enqueue_end)
    DevBuf tilectr;                          // two tile counters of render_r64_kernel, used by alternate launches
    DevBuf tstamp;                           // [2] %globaltimer: start of the message's render_r64_kernel, end of its finalize_kernel
    unsigned long long r64_count = 0;        // render_r64_kernel launches so far (picks the tile counter)
    bool after_fin = false;                  // the last thing this engine enqueued is a finalize_kernel (no event behind it)
    bool stamped = false;                    // the last enqueued render times itself with tstamp instead of ev0 / ev1
};

// SP_NO_PDL=1: launch render_r64_kernel and finalize_kernel in plain stream order and time messages with events (A/B runs)
static bool pdl_enabled()
{
    static const bool on = getenv("SP_NO_PDL") == nullptr;
    return on;
}

static thread_local std::string g_create_err;

static int fail(sp_engine *e, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (e) e->err = buf; else g_create_err = buf;
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _c = (call);                                                                   \
        if (_c != cudaSuccess) return fail(e, SP_E_CUDA, "%s: %s", #call, cudaGetErrorString(_c)); \
    } while (0)

static int ensure(sp_engine *e, DevBuf &b, size_t bytes)
{
    if (b.cap >= bytes && b.p) return SP_OK;
    if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    size_t want = (bytes + 255) & ~(size_t)255;
    if (want == 0) want = 256;
    cudaError_t c = cudaMalloc(&b.p, want);
    if (c != cudaSuccess) { b.p = nullptr; return fail(e, SP_E_CUDA, "cudaMalloc(%zu): %s", want, cudaGetErrorString(c)); }
    b.cap = want;
    return SP_OK;
}

// entry points other than sp_render work on the first device of a multi-device engine (taps, memory helpers, plan)
static sp_engine *dev0(sp_engine *e)
{
    if (e && !e->subs.empty()) { e->err.clear(); return e->subs[(size_t)e->cur]; }
    return e;
}

extern "C" const char *sp_last_error(sp_engine *e)
{
    if (!e) return g_create_err.c_str();
    if (!e->subs.empty() && e->err.empty()) return e->subs[(size_t)e->cur]->err.c_str();
    return e->err.c_str();
}

extern "C" int sp_create(sp_engine **out, const int *device_ids, int ndev)
{
    if (!out) return fail(nullptr, SP_E_INVAL, "sp_create: out is null");
    *out = nullptr;
    if (ndev < 1) ndev = 1;
    if (ndev > 1) {                          // one sub-engine per device; sp_render shards whole messages across them
        sp_engine *parent = new sp_engine();
        parent->ndev = ndev;
        for (int i = 0; i < ndev; i++) {
            sp_engine *sub = nullptr;
            const int d = device_ids ? device_ids[i] : i;
            const int rc = sp_create(&sub, &d, 1);
            if (rc) {
                for (sp_engine *s2 : parent->subs) sp_destroy(s2);
                delete parent;
                return rc;                   // g_create_err holds the message
            }
            parent->subs.push_back(sub);
        }
        parent->dev = parent->subs[0]->dev;
        parent->sm_count = parent->subs[0]->sm_count;
        // one communicator per device for the merge of device-resident shards (sp_render_shards).  A host without NCCL still
        // gets the engine: host-buffer messages are merged on the host, and sp_render_shards reports SP_E_NCCL.
        NcclApi *nc = nccl_api();
        if (!nc->lib) parent->nccl_err = nc->err;
        else {
            std::vector<int> devs;
            for (sp_engine *s2 : parent->subs) devs.push_back(s2->dev);
            parent->comms.assign((size_t)ndev, nullptr);
            const int r = nc->CommInitAll(parent->comms.data(), ndev, devs.data());
            if (r != 0) {
                parent->nccl_err = std::string("ncclCommInitAll: ") + (nc->GetErrorString ? nc->GetErrorString(r) : "failed");
                parent->comms.clear();
            }
        }
        *out = parent;
        return SP_OK;
    }
    int count = 0;
    cudaError_t c = cudaGetDeviceCount(&count);
    if (c != cudaSuccess || count == 0)
        return fail(nullptr, SP_E_NO_DEVICE, "no CUDA device (%s); this engine has no CPU fallback",
                    c != cudaSuccess ? cudaGetErrorString(c) : "device count is 0");
    const int dev = device_ids ? device_ids[0] : 0;
    if (dev < 0 || dev >= count) return fail(nullptr, SP_E_NO_DEVICE, "device %d out of range (count %d)", dev, count);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return fail(nullptr, SP_E_CUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10)
        return fail(nullptr, SP_E_NO_DEVICE, "device %d is sm_%d%d; kernels are built for sm_100a only (no fallback)", dev,
                    prop.major, prop.minor);
    sp_engine *e = new sp_engine();
    e->dev = dev;
    e->sm_count = prop.multiProcessorCount;
    if (cudaSetDevice(dev) != cudaSuccess || cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&e->ev0) != cudaSuccess || cudaEventCreate(&e->ev1) != cudaSuccess) {
        int rc = fail(nullptr, SP_E_CUDA, "stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
        delete e;
        return rc;
    }
    e->stream = e->own_stream;
    *out = e;
    return SP_OK;
}

extern "C" void sp_destroy(sp_engine *e)
{
    if (!e) return;
    if (!e->subs.empty()) {
        for (size_t g = 0; g < e->comms.size(); g++)
            if (e->comms[g]) { cudaSetDevice(e->subs[g]->dev); cudaDeviceSynchronize(); nccl_api()->CommDestroy(e->comms[g]); }
        for (sp_engine *sub : e->subs) sp_destroy(sub);
        delete e;
        return;
    }
    cudaSetDevice(e->dev);
    cudaDeviceSynchronize();
    for (auto &kv : e->tw) cudaFree(kv.second);
    DevBuf *bufs[] = { &e->in, &e->zin, &e->spec, &e->image, &e->fmin, &e->fmax, &e->fmid, &e->gauges, &e->hist, &e->jhist, &e->stats, &e->mm,
                       &e->lut, &e->window, &e->window_t, &e->acc, &e->jhtab, &e->ring, &e->ringctl, &e->scratch, &e->db, &e->synth_lut, &e->pin[0], &e->pin[1],
                       &e->pimg[0], &e->pimg[1], &e->tilectr, &e->tstamp };
    for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
    for (auto ev : e->prof0) cudaEventDestroy(ev);
    for (auto ev : e->prof1) cudaEventDestroy(ev);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    for (int i = 0; i < 2; i++) {
        if (e->ev_in[i]) cudaEventDestroy(e->ev_in[i]);
        if (e->ev_comp[i]) cudaEventDestroy(e->ev_comp[i]);
        if (e->ev_out[i]) cudaEventDestroy(e->ev_out[i]);
    }
    if (e->ev_setup) cudaEventDestroy(e->ev_setup);
    for (auto &s : e->inflight) {
        if (s.done) cudaEventDestroy(s.done);
        if (s.reply) cudaEventDestroy(s.reply);
        if (s.bounce) cudaFreeHost(s.bounce);
    }
    if (e->s_done) cudaStreamDestroy(e->s_done);
    if (e->s_h2d) cudaStreamDestroy(e->s_h2d);
    if (e->s_d2h) cudaStreamDestroy(e->s_d2h);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    delete e;
}

extern "C" int sp_set_stream(sp_engine *e, void *cuda_stream)
{
    e = dev0(e);
    if (!e) return SP_E_INVAL;
    e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
    return SP_OK;
}
extern "C" int sp_device_count(sp_engine *e) { return e ? e->ndev : 0; }
extern "C" int sp_select_device(sp_engine *e, int index)
{
    if (!e) return SP_E_INVAL;
    if (index < 0 || index >= e->ndev) return fail(e, SP_E_INVAL, "device index %d outside [0, %d)", index, e->ndev);
    e->cur = index;
    return SP_OK;
}
extern "C" int sp_sm_count(sp_engine *e) { return e ? e->sm_count : 0; }

// ------------------------------------------------------------------ helpers
static int ilog2_exact(int n)
{
    for (int i = 0; i < 31; i++) if ((1 << i) == n) return i;
    return -1;
}

// The samples that global frames [x0, x0 + count) read, as a piece of a buffer that starts at sample buf_first and holds
// byte_length bytes: sample s0 and bytes [b0, b1) of the buffer.  The start is rounded down to 16 samples (any format's byte
// offset stays 16-byte aligned), the end is the last frame's start + n.  The piece takes the samples its frames read and nothing
// more: a shard's buffer may extend past its frames (a caller may pass the whole capture with a frame sub-range).  The ragged tail
// (< 1 sample, or whatever lies between the last frame and the end of the capture) travels only with the piece that holds the
// message's last frame (msg_last).
struct Span { long long s0; unsigned long long b0, b1; };
static Span frame_span(double stride, int n, int sw, long long x0, long long count, long long buf_first, unsigned long long byte_length,
                       bool msg_last)
{
    long long s0 = sp::frame_pos(stride, x0);
    const long long s1 = sp::frame_pos(stride, x0 + count - 1) + n;
    s0 -= s0 % 16;
    if (s0 < buf_first) s0 = buf_first;
    unsigned long long b0 = (unsigned long long)(s0 - buf_first) * sw, b1 = (unsigned long long)(s1 - buf_first) * sw;
    if (b1 > byte_length || msg_last) b1 = byte_length;
    if (b0 > b1) b0 = b1;
    return { s0, b0, b1 };
}

static int upload_table(sp_engine *e, std::pair<Tw, int> key, const std::vector<float2> &h, const float2 **out)
{
    float2 *d = nullptr;
    CU(cudaMalloc(&d, sizeof(float2) * h.size()));
    CU(cudaMemcpyAsync(d, h.data(), sizeof(float2) * h.size(), cudaMemcpyHostToDevice, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->tw[key] = d;
    *out = d;
    return SP_OK;
}
static inline float2 twid(long long num, long long den)   // exp(-2 pi j num / den), double -> fp32 once
{
    const double a = 2.0 * M_PI * (double)(num % den) / (double)den;
    return make_float2((float)cos(a), (float)-sin(a));
}
// The table of one kind for size n, built and uploaded on first use:
//   big    [R-1][4096]  W_n^{j*k}, k = 1 .. R-1, j fastest      pre-passes of the four-step sizes, n = R * 4096: render_big_kernel
//                                                               and prepass_kernel (coalesced loads)
//   passA  [15][n/16]   W_n^{t*k}, k = 1 .. 15                  render_kernel, n >= 32
//   passB  [15][n/256]  W_{n/16}^{b*k}, k = 1 .. 15             render_kernel, n >= 512
//   tw14   [n/64][14]   W_n^{t*k}, k = 1 .. 7, 8, 16, .., 56    render_r64_kernel (n = 4096), render_rc_kernel (n = 2048)
//   w      [P][n/P]     W_n^{t*k}, k = 0 .. P-1                 render_w_kernel (P from w_log2p)
static int get_table(sp_engine *e, Tw kind, int n, const float2 **out)
{
    auto it = e->tw.find({ kind, n });
    if (it != e->tw.end()) { *out = it->second; return SP_OK; }
    std::vector<float2> h;
    switch (kind) {
    case Tw::big: {
        const int R = n / 4096;
        h.resize((size_t)(R - 1) * 4096);
        for (int k = 1; k < R; k++) for (int j = 0; j < 4096; j++) h[(size_t)(k - 1) * 4096 + j] = twid((long long)j * k, n);
        break;
    }
    case Tw::passA: {
        const int T = n / 16;
        h.resize((size_t)15 * T);
        for (int k = 1; k < 16; k++) for (int t = 0; t < T; t++) h[(size_t)(k - 1) * T + t] = twid((long long)t * k, n);
        break;
    }
    case Tw::passB: {
        const int RL = n / 256, N1 = n / 16;
        h.resize((size_t)15 * RL);
        for (int k = 1; k < 16; k++) for (int b = 0; b < RL; b++) h[(size_t)(k - 1) * RL + b] = twid((long long)b * k, N1);
        break;
    }
    case Tw::tw14: {
        static const int ks[14] = { 1, 2, 3, 4, 5, 6, 7, 8, 16, 24, 32, 40, 48, 56 };
        const int c = n / 64;
        h.resize((size_t)c * 14);
        for (int t = 0; t < c; t++) for (int i = 0; i < 14; i++) h[(size_t)t * 14 + i] = twid((long long)t * ks[i], n);
        break;
    }
    case Tw::w: {
        const int P = 1 << sp::w_log2p(ilog2_exact(n)), T = n / P;
        h.resize((size_t)n);
        for (int k = 0; k < P; k++) for (int t = 0; t < T; t++) h[(size_t)k * T + t] = twid((long long)t * k, n);
        break;
    }
    }
    return upload_table(e, { kind, n }, h, out);
}
// render_kernel's pass tables; null for the sizes that need none
static int get_pass_tables(sp_engine *e, int log2k, const float2 **twA, const float2 **twB)
{
    *twA = *twB = nullptr;
    int rc = SP_OK;
    if (log2k > 4) rc = get_table(e, Tw::passA, 1 << log2k, twA);
    if (!rc && log2k > 8) rc = get_table(e, Tw::passB, 1 << log2k, twB);
    return rc;
}

struct Plan {
    int log2k = 0;       // kernel FFT size (log2)
    int sub_r = 1;       // pre-pass radix (n = sub_r * 4096 when > 1)
    int tile = 0;        // frames per CTA tile
    int smem_x = 0;      // exchange area in float2
};

template <int L> static void fill_cfg(Plan &pl)
{
    pl.tile = sp::Cfg<L>::TILE;
    pl.smem_x = sp::Cfg<L>::SMEM_X;
}
static Plan make_plan(int log2n)
{
    Plan pl;
    if (log2n > 12) { pl.log2k = 12; pl.sub_r = 1 << (log2n - 12); } else pl.log2k = log2n;
    switch (pl.log2k) {
    case 1: fill_cfg<1>(pl); break;   case 2: fill_cfg<2>(pl); break;
    case 3: fill_cfg<3>(pl); break;   case 4: fill_cfg<4>(pl); break;   case 5: fill_cfg<5>(pl); break;
    case 6: fill_cfg<6>(pl); break;   case 7: fill_cfg<7>(pl); break;   case 8: fill_cfg<8>(pl); break;
    case 9: fill_cfg<9>(pl); break;   case 10: fill_cfg<10>(pl); break; case 11: fill_cfg<11>(pl); break;
    default: fill_cfg<12>(pl); break;
    }
    if (pl.sub_r > 1) pl.tile = 8;    // sub-frame tiles: 8 frames x one sub-sequence
    return pl;
}

// The fused kernel that takes the bulk of the frames described by p.  render_kernel (for n > 4096: prepass_kernel and the
// sub-frame render_kernel) takes whatever it leaves.  Every fused kernel writes a colour image with 4-byte-aligned rows (any width:
// rows that are not 32-byte aligned are written word by word) and at most 256 colours, and starts on a group of 8 frames, so the
// same frames take the same kernel whether a message is rendered in one piece, in pipeline chunks or in shards.
// For n > 4096 the frame count picks one of the two forms of the four-step transform (enqueue_frames).
enum class Route { none, r64, w, rc, fourstep };
static Route route(const Plan &pl, int fmt, const Params &p)
{
    const sp::Kernels &k = kernels_for(fmt);
    if (!p.image || p.db_out || p.cmap_len > 256 || p.chunk_first % 8 != 0 || ((uintptr_t)p.image & 3) != 0) return Route::none;
    if (pl.sub_r > 1) return !p.waterfall && !p.channel_mode && k.big ? Route::fourstep : Route::none;
    if (sp::sample_width(fmt) > 8) return Route::none;           // a raw frame must fit the exchange buffer
    // r64 and w: waterfall rows in the store warps, split-real in the FFT warps
    if (pl.log2k == 12 && k.r64) return Route::r64;
    if (pl.log2k >= 6 && pl.log2k <= 10 && k.w) return Route::w;
    if (pl.log2k == 11 && k.rc && !p.channel_mode) return Route::rc;
    return Route::none;
}

extern "C" const char *sp_kernel_plan(sp_engine *e, int format, int n, int channel_mode)
{
    e = dev0(e);
    if (!e) return "";
    const int l = ilog2_exact(n);
    char buf[640];
    if (l < 1 || l > 18 || format < 0 || format >= SP_FORMAT_COUNT) { e->plan = "unsupported"; return e->plan.c_str(); }
    Plan pl = make_plan(l);
    const char *fname = specialised(format) ? k_names[format] : "runtime-format";
    Params p;                                                   // spectrogram layout, 256 colours, an aligned image, no dB tap
    memset(&p, 0, sizeof p);
    p.image = (uint8_t *)(uintptr_t)256;
    p.cmap_len = 256;
    p.channel_mode = channel_mode ? 1 : 0;
    const int P = pl.log2k <= 6 ? 8 : (pl.log2k <= 8 ? 16 : 32);
    size_t o = 0;
    // the kernel the bulk of the message takes, then what catches the rest
    switch (route(pl, format, p)) {
    case Route::fourstep:
        o += snprintf(buf + o, sizeof buf - o, "four-step n = %d x 4096: render_big_kernel<%s> (one persistent launch, pre-pass and 64x64 second stage as queue items over an "
                      "L2-resident ring; long captures at n = 32768 / 65536, SP_FOURSTEP=ring) or prepass_kernel + render_r64_kernel<sub-frame> over an HBM scratch | ",
                      pl.sub_r, fname);
        break;
    case Route::r64:
        o += snprintf(buf + o, sizeof buf - o, "render_r64_kernel<%s> (64x64 FFT, one exchange, 4 frame streams + store warpgroup, TMA-staged input, joint histogram, "
                      "RGBA tiles + tensor-TMA row stores%s) | ", fname, channel_mode ? ", split-real in the FFT warps" : "");
        break;
    case Route::w:
        o += snprintf(buf + o, sizeof buf - o, "render_w_kernel<%s, N=%dx%d> (warp-synchronous, one exchange, span-staged input, tables in registers, joint histogram, "
                      "store warpgroup, spectrogram and waterfall layout%s) | ", fname, P, (1 << pl.log2k) / P, channel_mode ? ", split-real in the FFT warps" : "");
        break;
    case Route::rc:
        o += snprintf(buf + o, sizeof buf - o, "render_rc_kernel<%s, N=64x%d> (one exchange, joint histogram, TMA-staged input, store warpgroup) | ", fname, (1 << pl.log2k) / 64);
        break;
    case Route::none: break;
    }
    snprintf(buf + o, sizeof buf - o, "%s%srender_kernel<N=%d,%s> tile=%d frames%s (every option; remainder frames, ragged ends, dB tap, cmap_len > 256)",
             pl.sub_r > 1 ? "prepass_kernel<R=" : "", pl.sub_r > 1 ? (std::to_string(pl.sub_r) + "> + ").c_str() : "", 1 << pl.log2k, fname, pl.tile,
             channel_mode ? " +splitreal" : "");
    e->plan = buf;
    return e->plan.c_str();
}

// Everything a render needs on the device, resolved from a request.
struct Job {
    Params p;
    Plan plan;
    int log2n = 0;
    long long width = 0;       // local frames
    double range = 0, gain = 0;
    uint8_t *d_image = nullptr;
    uint8_t *d_gmin = nullptr, *d_gmax = nullptr, *d_gamp = nullptr;
    unsigned long long *d_cb = nullptr, *d_c = nullptr;
    double *d_stats = nullptr;
    bool pipelined = false;    // host buffers streamed chunk by chunk: no whole-message device copies
    bool pdl = false;          // the render kernel may start early behind the previous message's finalize_kernel
    bool stamp = false;        // device time from tstamp (the message goes through render_r64_kernel) instead of ev0 / ev1
};

// bracket a render-kernel launch with the next event pair of the profiling ring.  An event pair between two dependent kernels
// costs the stream several microseconds (the next launch can no longer be queued behind the running kernel), so only every
// prof_every-th launch is bracketed (sp_profile_enable's `every`, default 1): the ring then holds a sample of the launches.
static void prof_begin(sp_engine *e)
{
    e->prof_this = !e->prof0.empty() && (e->prof_seq++ % (long long)e->prof_every) == 0;
    if (e->prof_this) cudaEventRecord(e->prof0[e->prof_count % (long long)e->prof0.size()], e->stream);
}
static void prof_end(sp_engine *e)
{
    if (e->prof_this) { cudaEventRecord(e->prof1[e->prof_count % (long long)e->prof1.size()], e->stream); e->prof_count++; }
}

static int validate(sp_engine *e, const sp_request *rq, bool shard, double *sample_count, double *stride)
{
    if (!rq->buffer || !rq->windowc || !rq->cmap_rgb) return fail(e, SP_E_INVAL, "buffer, windowc and cmap_rgb are required");
    if (rq->format < 0 || rq->format >= SP_FORMAT_COUNT) return fail(e, SP_E_BAD_FORMAT, "format %d out of range", rq->format);
    const int l = ilog2_exact(rq->n);
    if (l < 0) return fail(e, SP_E_BAD_N, "Length is not a power of 2");          // lib/fft_nayuki.js:39
    if (rq->n < SP_MIN_N || rq->n > SP_MAX_N) return fail(e, SP_E_BAD_N, "n=%d outside [%d, %d]", rq->n, SP_MIN_N, SP_MAX_N);
    if (rq->cmap_len < 2 || rq->cmap_len > SP_MAX_CMAP) return fail(e, SP_E_BAD_CMAP, "cmap_len=%d outside [2, %d]", rq->cmap_len, SP_MAX_CMAP);
    const uint64_t total_bytes = shard ? rq->total_byte_length : rq->byte_length;
    const int64_t total_width = shard ? rq->total_width : rq->width;
    if (total_bytes % (uint64_t)sp::element_size(rq->format))
        return fail(e, SP_E_RAGGED, "byte length %llu is not a multiple of the %d-byte element size (typed array construction throws)",
                    (unsigned long long)total_bytes, sp::element_size(rq->format));
    if (total_width < 1 || rq->width < 1) return fail(e, SP_E_BAD_WIDTH, "width=%lld", (long long)(total_width < 1 ? total_width : rq->width));
    const double sc = (double)total_bytes / (double)sp::sample_width(rq->format);   // lib/samples.js:167
    // A capture shorter than one frame is answered like the reference answers it (it never throws): every frame reads
    // `undefined` past the typed array and comes out as NaN / colour 0 through the bounds-checked decode.  Only a shard
    // of such a message is refused (there is nothing to shard).
    if (sc < (double)rq->n && shard) return fail(e, SP_E_TOO_SHORT, "sampleCount %.1f < n %d in a sharded message", sc, rq->n);
    if (!(rq->range != 0.0) || !std::isfinite(rq->range) || !std::isfinite(rq->gain) || !(rq->block_norm > 0.0))
        return fail(e, SP_E_INVAL, "range must be finite and non-zero, gain finite, block_norm > 0");
    if (10.0 * log10(rq->block_norm) < -75.0)
        return fail(e, SP_E_INVAL, "block_norm %.3g is below -75 dB (1/weight of any window up to n = 65536 is above -49 dB)", rq->block_norm);
    *sample_count = sc;
    // lib/worker.js:50.  A one-frame message divides by zero there: stride is +-Infinity or NaN, stride * 0 is NaN and
    // ~~(0.5 + NaN) == 0, i.e. the frame starts at sample 0 - the same as stride 0.
    *stride = total_width == 1 ? 0.0 : (sc - (double)rq->n) / (double)(total_width - 1);
    if (shard) {
        if (rq->frame_first < 0 || rq->frame_first + rq->width > total_width)
            return fail(e, SP_E_RANGE, "frame range [%lld, %lld) outside total width %lld", (long long)rq->frame_first,
                        (long long)(rq->frame_first + rq->width), (long long)total_width);
        // the shard buffer must cover every sample its frames read
        const long long p_first = sp::frame_pos(*stride, rq->frame_first);
        const long long p_last = sp::frame_pos(*stride, rq->frame_first + rq->width - 1) + rq->n;
        const long long have_first = (long long)rq->buffer_first_sample;
        const double have_last = (double)have_first + (double)rq->byte_length / sp::sample_width(rq->format);
        if (p_first < have_first || ((double)p_last > have_last && (double)p_last <= sc))
            return fail(e, SP_E_RANGE, "shard buffer [%lld, %.0f) does not cover samples [%lld, %lld) needed by its frames",
                        have_first, have_last, p_first, p_last);
    }
    return SP_OK;
}

// Build the device-side job: upload constants, bind buffers.
// Give the L2 back: render_big_kernel pins its pre-pass ring with a persisting access-policy window, and the set-aside half of the
// cache is not available to normal lines while it stands (every other kernel runs 5 - 35 % slower under it).
static void release_l2_window(sp_engine *e)
{
    if (!e->l2_window) return;
    cudaStreamAttrValue av;
    memset(&av, 0, sizeof av);
    cudaStreamSetAttribute(e->stream, cudaStreamAttributeAccessPolicyWindow, &av);
    cudaCtxResetPersistingL2Cache();
    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0);
    cudaGetLastError();
    e->l2_window = 0;
}

static int prepare(sp_engine *e, const sp_request *rq, sp_reply *rp, Job &j, bool want_db, float *db_dev)
{
    const bool shard = rq->total_width != 0 || rq->total_byte_length != 0;
    double sample_count = 0, stride = 0;
    int rc = validate(e, rq, shard, &sample_count, &stride);
    if (rc) return rc;
    CU(cudaSetDevice(e->dev));
    // a render may overlap the previous message's finalize_kernel only when nothing was enqueued in between: a copy below
    // (input, window, LUT) or one in enqueue_begin clears j.pdl
    j.pdl = e->after_fin;
    e->after_fin = false;
    const int n = rq->n;
    j.log2n = ilog2_exact(n);
    j.plan = make_plan(j.log2n);
    if (j.plan.sub_r == 1) release_l2_window(e);          // the last render may have pinned the pre-pass ring of render_big_kernel in L2
    j.width = rq->width;
    j.range = rq->range;
    j.gain = rq->gain;
    const bool in_dev = rq->flags & SP_F_BUFFER_ON_DEVICE, out_dev = rq->flags & SP_F_REPLY_ON_DEVICE;
    Params &p = j.p;
    memset(&p, 0, sizeof p);

    // ---- input bytes
    if (in_dev) {
        if ((uintptr_t)rq->buffer & 15) return fail(e, SP_E_ALIGN, "device buffer must be 16-byte aligned");
        p.buf = (const uint8_t *)rq->buffer;
    } else if (j.pipelined) {
        p.buf = nullptr;                                   // set per chunk by render_pipelined
    } else {
        if ((rc = ensure(e, e->in, rq->byte_length + 16))) return rc;
        CU(cudaMemcpyAsync(e->in.p, rq->buffer, rq->byte_length, cudaMemcpyHostToDevice, e->stream));
        p.buf = (const uint8_t *)e->in.p;
        j.pdl = false;
    }
    p.valid_bytes = rq->byte_length;
    p.sample_base = shard ? (long long)rq->buffer_first_sample : 0;
    p.format = rq->format;
    p.n_full = n;
    p.stride = stride;
    p.frame_first = shard ? rq->frame_first : 0;
    p.nframes = rq->width;
    p.chunk_first = 0;
    p.chunk_frames = rq->width;

    // ---- window (fp32, rounded once), colour LUT, twiddles.  Uploaded only when they change, from
    // engine-owned staging vectors, so a steady stream of messages never synchronises the host here.
    {
        // power-of-two sample scales are folded into the fp32 window (exact), see decode_raw()
        const float wscale = specialised(rq->format) ? sp::raw_scale_rt(rq->format) : 1.0f;
        bool same_w = e->h_window.size() == (size_t)n;
        if (same_w)
            for (int i = 0; i < n; i++) if (e->h_window[i] != (float)rq->windowc[i] * wscale) { same_w = false; break; }
        bool same_l = e->h_lut.size() == (size_t)rq->cmap_len;
        if (same_l)
            for (int i = 0; i < rq->cmap_len; i++) {
                const uint32_t v = (uint32_t)rq->cmap_rgb[3 * i] | ((uint32_t)rq->cmap_rgb[3 * i + 1] << 8) |
                                   ((uint32_t)rq->cmap_rgb[3 * i + 2] << 16) | 0xff000000u;
                if (e->h_lut[i] != v) { same_l = false; break; }
            }
        if (!same_w || !same_l) {
            CU(cudaStreamSynchronize(e->stream));                       // staging vectors may still be in flight
            j.pdl = false;
        }
        if (!same_w) {
            e->h_window.resize((size_t)n);
            for (int i = 0; i < n; i++) e->h_window[i] = (float)rq->windowc[i] * wscale;
            if ((rc = ensure(e, e->window, sizeof(float) * (size_t)n))) return rc;
            CU(cudaMemcpyAsync(e->window.p, e->h_window.data(), sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, e->stream));
            if (n == 4096) {
                // render_r64_kernel reads its 64 coefficients per thread straight from global memory (L1-resident): [16][64] float4,
                // element (q, t) = w[64*(4q + i) + t], so that a warp's LDG.128 covers 512 contiguous bytes
                e->h_window_t.resize(4096);
                for (int q = 0; q < 16; q++) for (int t = 0; t < 64; t++) for (int i = 0; i < 4; i++)
                    e->h_window_t[(size_t)(q * 64 + t) * 4 + i] = e->h_window[(size_t)64 * (4 * q + i) + t];
                if ((rc = ensure(e, e->window_t, sizeof(float) * 4096))) return rc;
                CU(cudaMemcpyAsync(e->window_t.p, e->h_window_t.data(), sizeof(float) * 4096, cudaMemcpyHostToDevice, e->stream));
            }
        }
        if (!same_l) {
            e->h_lut.resize((size_t)rq->cmap_len);
            for (int i = 0; i < rq->cmap_len; i++)          // R, G, B, A=255 in memory order (lib/worker.js:118-121)
                e->h_lut[i] = (uint32_t)rq->cmap_rgb[3 * i] | ((uint32_t)rq->cmap_rgb[3 * i + 1] << 8) |
                              ((uint32_t)rq->cmap_rgb[3 * i + 2] << 16) | 0xff000000u;
            if ((rc = ensure(e, e->lut, sizeof(uint32_t) * (size_t)rq->cmap_len))) return rc;
            CU(cudaMemcpyAsync(e->lut.p, e->h_lut.data(), sizeof(uint32_t) * (size_t)rq->cmap_len, cudaMemcpyHostToDevice, e->stream));
        }
    }
    p.window = (const float *)e->window.p;
    p.window_t = (const float4 *)e->window_t.p;
    p.lut = (const uint32_t *)e->lut.p;
    if ((rc = get_pass_tables(e, j.plan.log2k, &p.twA, &p.twB))) return rc;

    // ---- dB / colour constants (lib/worker.js:32,39,93,111)
    const double block_norm_db = 10.0 * log10(rq->block_norm);
    const double color_norm = (double)rq->cmap_len / -rq->range;
    p.c0 = (float)block_norm_db;
    p.c1 = (float)(5.0 * log10(2.0));
    p.gn = (float)(-color_norm);                                    // grayU = cmax - (d0 + gain) * color_norm
    p.gc = (float)((double)(rq->cmap_len - 1) - rq->gain * color_norm);
    p.cmaxf = (float)(rq->cmap_len - 1);
    p.cmap_len = rq->cmap_len;
    {   // joint-histogram constants (sp_kernels.cuh, jh_eval): in double, rounded once
        const double c1 = 5.0 * log10(2.0), cmaxd = (double)(rq->cmap_len - 1);
        p.jA = (float)(-10.0 * c1 / sp::JH_RCAP);
        p.jB = (float)((2.5 - 10.0 * block_norm_db) / sp::JH_RCAP);
        p.jC = (float)(-color_norm * c1 / cmaxd);
        p.jD = (float)((cmaxd - (block_norm_db + rq->gain) * color_norm) / cmaxd);
    }
    p.waterfall = rq->waterfall ? 1 : 0;
    p.channel_mode = rq->channel_mode ? 1 : 0;
    p.sub_r = j.plan.sub_r;

    // ---- outputs
    const size_t W = (size_t)rq->width;
    const bool want_image = rp->image && !(rq->flags & SP_F_NO_IMAGE) && !want_db;
    if (want_image) {
        if (out_dev) {
            j.d_image = rp->image;
        } else if (j.pipelined) {
            j.d_image = (uint8_t *)(uintptr_t)16;              // placeholder: per-chunk tiles (render_pipelined)
        } else {
            if ((rc = ensure(e, e->image, 4 * W * (size_t)n))) return rc;
            j.d_image = (uint8_t *)e->image.p;
        }
    }
    p.image = j.d_image;
    if ((rc = ensure(e, e->fmin, 4 * W)) || (rc = ensure(e, e->fmax, 4 * W)) || (rc = ensure(e, e->fmid, 8 * W))) return rc;
    p.fmin = (float *)e->fmin.p;
    p.fmax = (float *)e->fmax.p;
    p.fmid = (float2 *)e->fmid.p;
    if ((rc = ensure(e, e->hist, 8 * (size_t)(SP_CB_HIST_SIZE + SP_MAX_CMAP)))) return rc;
    if ((rc = ensure(e, e->stats, 16)) || (rc = ensure(e, e->mm, 16)) || (rc = ensure(e, e->jhist, 8 * (size_t)sp::JH_SIZE))) return rc;
    p.j_hist = (unsigned long long *)e->jhist.p;
    if ((rc = ensure(e, e->gauges, 3 * W))) return rc;
    if (out_dev) {
        j.d_cb = rp->cB_hist ? (unsigned long long *)rp->cB_hist : (unsigned long long *)e->hist.p;
        j.d_c = rp->c_hist ? (unsigned long long *)rp->c_hist : (unsigned long long *)e->hist.p + SP_CB_HIST_SIZE;
        j.d_gmin = rp->gauge_mins; j.d_gmax = rp->gauge_maxs; j.d_gamp = rp->gauge_amps;
    } else {
        j.d_cb = (unsigned long long *)e->hist.p;
        j.d_c = (unsigned long long *)e->hist.p + SP_CB_HIST_SIZE;
        j.d_gmin = (uint8_t *)e->gauges.p; j.d_gmax = j.d_gmin + W; j.d_gamp = j.d_gmax + W;
    }
    // the kernels accumulate into engine-owned counters; finalize_kernel copies them to the reply (j.d_cb / j.d_c) and zeroes them
    if ((rc = ensure(e, e->acc, 8 * (size_t)(SP_CB_HIST_SIZE + SP_MAX_CMAP))) || (rc = ensure(e, e->jhtab, 8 * (size_t)sp::JH_BINS))) return rc;
    p.cb_hist = (unsigned long long *)e->acc.p;
    p.c_hist = (unsigned long long *)e->acc.p + SP_CB_HIST_SIZE;
    j.d_stats = (out_dev && rp->minmax_dev) ? rp->minmax_dev : (double *)e->stats.p;
    e->stats_src = j.d_stats;
    p.db_out = want_db ? db_dev : nullptr;
    return SP_OK;
}

// Tensor map of the [n rows][width] RGBA picture for the store warps of render_r64_kernel: boxes of 32 rows x 8 pixels,
// 32-byte swizzle.  The encoder is a driver entry point; it is resolved at run time so that the library keeps linking the
// CUDA runtime only.
typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static encode_tiled_fn tensor_map_encoder()
{
    static encode_tiled_fn fn = []() -> encode_tiled_fn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess) return nullptr;
        return (encode_tiled_fn)p;
    }();
    return fn;
}
static bool image_tensor_map(CUtensorMap *tm, uint8_t *image, long long width, int rows)
{
    encode_tiled_fn enc = tensor_map_encoder();
    if (!enc || !image || width % 8 != 0 || ((uintptr_t)image & 31) != 0 || width > 0x7fffffffLL) return false;
    const cuuint64_t dims[2] = { (cuuint64_t)width, (cuuint64_t)rows };
    const cuuint64_t strides[1] = { (cuuint64_t)width * 4 };
    const cuuint32_t box[2] = { 8, 32 }, estr[2] = { 1, 1 };
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, image, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The leading whole groups of 8 frames of the chunk q whose `len` samples lie inside the buffer: the same frames whatever the
// chunking or sharding, so pipelined / sharded renders stay bit-identical to the single shot.  The fused kernels stage raw frames
// in whole 16-byte units (sp::staged_extent), which the buffer's readable slack covers as long as the frame itself lies inside.
static long long frames_inside(const Params &q, int len)
{
    const int sw = sp::sample_width(q.format);
    auto inside = [&](long long xr) { return sp::samples_inside(sp::frame_start(q, xr), len, sw, q.valid_bytes); };
    long long nf = q.chunk_frames / 8 * 8;                 // the last tile may be partial (a multiple of 8 frames)
    while (nf > 0 && !inside(nf - 1)) nf -= 8;
    if (nf > 0 && !inside(0)) nf = 0;
    return nf;
}

// The launch every fused kernel shares, of frames [0, nf) of the chunk q.  launch(r, grid, occ_out) calls the format's launcher
// (occ_out set: occupancy probe only).  A kernel that does not fit an SM, or is not built for the format, takes no frames
// (*nfast stays 0) and the caller's remaining kernels take them.  Otherwise setup(r) does the family's own work on the launch's
// parameters, and the kernel runs ntiles tiles on at most one CTA per SM, in one slot of the profiling ring; `kernels` is what
// the launch adds to kernel_launches.
static int no_setup(Params &) { return SP_OK; }
template <typename Launch, typename Setup>
static int launch_fused(sp_engine *e, const Params &q, long long nf, long long ntiles, int kernels, long long *nfast, Launch launch, Setup setup)
{
    int occ = 0, rc;
    CU(launch(q, 0, &occ));
    if (occ < 1) return SP_OK;
    Params r = q;
    r.chunk_frames = nf;
    r.ntiles = ntiles;
    if ((rc = setup(r))) return rc;
    prof_begin(e);
    CU(launch(r, (int)(ntiles < e->sm_count ? ntiles : e->sm_count), nullptr));
    prof_end(e);
    e->launches += kernels;
    *nfast = nf;
    return SP_OK;
}

// render_r64_kernel: N = 4096, or in sub-frame mode the second stage of the HBM-scratch form of n > 4096, which reads the
// pre-pass scratch instead of the buffer and takes every whole group of 8 frames.  pdl: launch with programmatic stream
// serialization (the kernel ahead of it cannot write what the kernel reads before its griddep_wait); stamp: CTA 0 records the
// message's start time in tstamp[0].
static int launch_r64_kernel(sp_engine *e, const sp::Kernels &k, const Params &q, long long *nfast, bool pdl = false, bool stamp = false)
{
    const bool sub = q.sub_r > 1;
    const long long nf = sub ? q.chunk_frames / 8 * 8 : frames_inside(q, 4096);   // the last tile may be partial (8 of 16 frames)
    if (nf == 0) return SP_OK;
    const float2 *tw14 = nullptr;
    int rc = get_table(e, Tw::tw14, 4096, &tw14);
    if (rc) return rc;
    CUtensorMap tm;
    memset(&tm, 0, sizeof tm);
    auto launch = [&](const Params &r, int grid, int *occ) { return k.r64(sub ? 1 : 0, &r, grid, e->stream, tw14, &tm, pdl ? 1 : 0, occ); };
    auto setup = [&](Params &r) -> int {
        if (!e->tilectr.p) {                               // the kernel leaves its counter at zero: set once
            if ((rc = ensure(e, e->tilectr, 16))) return rc;
            CU(cudaMemsetAsync(e->tilectr.p, 0, 16, e->stream));
            pdl = false;
        }
        if (stamp && (rc = ensure(e, e->tstamp, 16))) return rc;
        r.use_tma = (!sub && !r.waterfall && image_tensor_map(&tm, r.image, r.nframes, r.n_full)) ? 1 : 0;
        r.tile_ctr = (unsigned long long *)e->tilectr.p + (e->r64_count++ & 1);
        r.t_stamp = stamp ? (unsigned long long *)e->tstamp.p : nullptr;
        return SP_OK;
    };
    return launch_fused(e, q, nf, ((nf + 15) / 16) * (sub ? q.sub_r : 1), 1, nfast, launch, setup);
}

// n = R * 4096: ONE launch of render_big_kernel (a pre-pass and a second stage, counted as two kernels), whose pre-pass output
// lives in an L2-resident ring of S blocks (S * 8 * n * 8 bytes, pinned by a persisting access-policy window).  The kernel is
// persistent and takes its work from a queue: one CTA per SM.
static int launch_big_kernel(sp_engine *e, const sp::Kernels &k, const Params &q, long long *nfast)
{
    const int n = q.n_full, R = q.sub_r;
    const long long nf = frames_inside(q, n);
    if (nf == 0) return SP_OK;
    sp::BigArgs g;
    memset(&g, 0, sizeof g);
    const float2 *tw14 = nullptr;
    auto launch = [&](const Params &r, int grid, int *occ) { return k.big(&r, &g, grid, e->stream, tw14, occ); };
    auto setup = [&](Params &) -> int {
        int rc;
        const int env_slots = getenv("SP_BIG_SLOTS") ? atoi(getenv("SP_BIG_SLOTS")) : 0;       // tuning / tests: ring slots and pre-pass lead
        const int env_lead = getenv("SP_BIG_LEAD") ? atoi(getenv("SP_BIG_LEAD")) : 0;
        // Ring: 64 MB, half of the L2 (every CTA holds 512 KB of it for the length of a second-stage tile: with less the pre-pass
        // waits for free slots, with more the ring no longer fits the 79 MB that can be pinned and spills to HBM - ncu: 1.0 x the
        // algorithmic DRAM traffic at 64 MB, 1.23 x at 80 MB; profiles/r02_big_kernel.txt), at least 8 blocks; the pre-pass runs
        // L = 3 S / 8 blocks ahead of the second stage.
        const size_t block_bytes = (size_t)8 * (size_t)n * 8;
        int S = env_slots > 0 ? env_slots : (int)(((size_t)64 << 20) / block_bytes);
        if (S < 8 && env_slots <= 0) S = 8;
        if (S < 2) S = 2;
        if (S > 64) S = 64;
        int L = env_lead > 0 ? env_lead : (3 * S / 8 > 2 ? 3 * S / 8 : 2);
        if (L > S) L = S;
        if (L < 1) L = 1;
        const float2 *twT = nullptr;
        // ringctl: BigArgs::ctl for up to 64 slots, then BigArgs::stats at the next 64-byte boundary
        const size_t ctl_bytes = 4 * (size_t)(1 + 2 * 64), stats_off = (ctl_bytes + 63) & ~(size_t)63;
        if ((rc = get_table(e, Tw::tw14, 4096, &tw14)) || (rc = get_table(e, Tw::big, n, &twT))) return rc;
        if ((rc = ensure(e, e->ring, (size_t)S * block_bytes)) || (rc = ensure(e, e->ringctl, stats_off + 64))) return rc;
        if (e->l2_window != (size_t)S * block_bytes) {
            // keep the ring in L2: persisting lines for the ring's address range, everything else streams through the rest
            cudaDeviceProp prop;
            CU(cudaGetDeviceProperties(&prop, e->dev));
            size_t want = (size_t)S * block_bytes;
            if (prop.persistingL2CacheMaxSize > 0) {
                const size_t set_aside = want < (size_t)prop.persistingL2CacheMaxSize ? want : (size_t)prop.persistingL2CacheMaxSize;
                cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside);
                cudaStreamAttrValue av;
                memset(&av, 0, sizeof av);
                av.accessPolicyWindow.base_ptr = e->ring.p;
                av.accessPolicyWindow.num_bytes = want < (size_t)prop.accessPolicyMaxWindowSize ? want : (size_t)prop.accessPolicyMaxWindowSize;
                av.accessPolicyWindow.hitRatio = 1.0f;
                av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
                av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
                cudaStreamSetAttribute(e->stream, cudaStreamAttributeAccessPolicyWindow, &av);
                cudaGetLastError();                               // best effort: the kernel is correct without the pin
            }
            e->l2_window = want;
        }
        CU(cudaMemsetAsync(e->ringctl.p, 0, ctl_bytes, e->stream));
        g.ring = (float2 *)e->ring.p;
        g.twT = twT;
        g.ctl = (unsigned *)e->ringctl.p;
        g.slots = S;
        g.lead = L;
        g.nblocks = nf / 8;
        g.R = R;
        // SP_BIG_STATS=1: per-phase SM cycle sums of the launch (development), printed at the next launch
        static const bool want_stats = getenv("SP_BIG_STATS") != nullptr;
        if (want_stats) {
            g.stats = (unsigned long long *)((unsigned char *)e->ringctl.p + stats_off);
            unsigned long long h[6];
            CU(cudaMemcpyAsync(h, g.stats, sizeof h, cudaMemcpyDeviceToHost, e->stream));   // the PREVIOUS launch's sums (stream order)
            CU(cudaStreamSynchronize(e->stream));
            if (h[4] || h[5])
                fprintf(stderr, "[big] P: %llu items, wait %.0f work %.0f cycles/item | F: %llu tiles, wait %.0f work %.0f cycles/tile\n", h[4],
                        h[4] ? (double)h[0] / h[4] : 0.0, h[4] ? (double)h[1] / h[4] : 0.0, h[5], h[5] ? (double)h[2] / h[5] : 0.0, h[5] ? (double)h[3] / h[5] : 0.0);
            CU(cudaMemsetAsync(g.stats, 0, sizeof h, e->stream));
        }
        return SP_OK;
    };
    return launch_fused(e, q, nf, e->sm_count, 2, nfast, launch, setup);
}

// render_w_kernel: N = 64 .. 1024
static int launch_w_kernel(sp_engine *e, const sp::Kernels &k, int log2n, const Params &q, long long *nfast)
{
    const int n = 1 << log2n, tile = sp::w_tile_frames(log2n);
    const long long nf = frames_inside(q, n);
    if (nf == 0) return SP_OK;
    const float2 *twW = nullptr;
    const int rc = get_table(e, Tw::w, n, &twW);
    if (rc) return rc;
    return launch_fused(e, q, nf, (nf + tile - 1) / tile, 1, nfast,
                        [&](const Params &r, int grid, int *occ) { return k.w(log2n, &r, grid, e->stream, twW, occ); }, no_setup);
}

// render_rc_kernel: N = 2048, tiles of 65536 / N frames
static int launch_rc_kernel(sp_engine *e, const sp::Kernels &k, int log2n, const Params &q, long long *nfast)
{
    const int n = 1 << log2n, tile = 65536 / n;
    const long long nf = frames_inside(q, n);
    if (nf == 0) return SP_OK;
    const float2 *tw14 = nullptr;
    const int rc = get_table(e, Tw::tw14, n, &tw14);
    if (rc) return rc;
    return launch_fused(e, q, nf, (nf + tile - 1) / tile, 1, nfast,
                        [&](const Params &r, int grid, int *occ) { return k.rc(log2n, &r, grid, e->stream, tw14, occ); }, no_setup);
}

// render_kernel (in sub-frame mode for n > 4096) over every frame of the chunk q, in one slot of the profiling ring.  It is the
// kernel that takes what the fused kernels leave, so unlike launch_fused a kernel that does not fit an SM is an error.
static int launch_render_kernel(sp_engine *e, const sp::Kernels &k, const Plan &pl, Params q)
{
    const size_t smem = sp::main_smem_bytes(pl.smem_x, q.cmap_len, pl.log2k > 8 ? 15 * ((1 << pl.log2k) / 256) : 0);
    int occ = 0;
    CU(k.render(pl.log2k, &q, 0, smem, e->stream, &occ));
    if (occ < 1) return fail(e, SP_E_CUDA, "render kernel does not fit an SM (smem %zu)", smem);
    q.ntiles = (q.chunk_frames + pl.tile - 1) / pl.tile * pl.sub_r;
    const long long cap = (long long)e->sm_count * occ;
    prof_begin(e);
    CU(k.render(pl.log2k, &q, (int)(q.ntiles < cap ? q.ntiles : cap), smem, e->stream, nullptr));
    prof_end(e);
    e->launches++;
    return SP_OK;
}

// Enqueue all kernels of a job on e->stream (bracketed by the timing events).
static int enqueue_begin(sp_engine *e, Job &j)
{
    e->launches = 0;
    // device time: a message whose frames go through render_r64_kernel is timed by that kernel and finalize_kernel
    // (%globaltimer), so that no event sits between the finalize_kernel of one message and the render of the next
    j.stamp = pdl_enabled() && !j.pipelined && route(j.plan, j.p.format, j.p) == Route::r64;
    if (e->acc_dirty) {
        j.pdl = false;
        // first render, or the previous one was abandoned before finalize_kernel could clean up: zero every accumulator once
        const unsigned mm0[4] = { 0x80000000u /* f2ord(0.0f) */, 0x3cb7ffffu /* f2ord(-200.0f) */, 0u, 0u };
        CU(cudaMemsetAsync(e->acc.p, 0, 8 * (size_t)(SP_CB_HIST_SIZE + SP_MAX_CMAP), e->stream));
        CU(cudaMemsetAsync(e->jhist.p, 0, 8 * (size_t)sp::JH_SIZE, e->stream));
        CU(cudaMemcpyAsync(e->mm.p, mm0, 16, cudaMemcpyHostToDevice, e->stream));
        CU(cudaStreamSynchronize(e->stream));                 // (mm0 lives on this stack frame)
    }
    e->acc_dirty = true;                                      // until finalize_kernel of THIS render has been enqueued
    // decode table of the joint histogram: rebuilt only when the dB / colour constants change
    const float key[5] = { j.p.jA, j.p.jB, j.p.jC, j.p.jD, (float)j.p.cmap_len };
    if (memcmp(key, e->jhtab_key, sizeof key)) {
        sp::jh_table_kernel<<<(sp::JH_BINS + 255) / 256, 256, 0, e->stream>>>(sp::jh_const(j.p), j.p.cmap_len - 1, (int2 *)e->jhtab.p);
        memcpy(e->jhtab_key, key, sizeof key);
        e->launches++;
        j.pdl = false;
    }
    if (!j.stamp) CU(cudaEventRecord(e->ev0, e->stream));
    e->stamped = j.stamp;
    return SP_OK;
}

// the render kernels for the frames described by p (a whole message, a shard, or one pipeline chunk)
static int enqueue_frames(sp_engine *e, Job &j, Params &p)
{
    const int fmt = p.format;
    const sp::Kernels &k = kernels_for(fmt);
    const Route fused = route(j.plan, fmt, p);
    if (j.plan.sub_r == 1) {
        Params q = p;
        long long nfast = 0;
        int rc = SP_OK;
        if (fused == Route::r64) rc = launch_r64_kernel(e, k, q, &nfast, j.pdl && pdl_enabled(), j.stamp);
        else if (fused == Route::w) rc = launch_w_kernel(e, k, j.plan.log2k, q, &nfast);
        else if (fused == Route::rc) rc = launch_rc_kernel(e, k, j.plan.log2k, q, &nfast);
        if (rc) return rc;
        q.chunk_first += nfast;
        q.chunk_frames -= nfast;
        if (j.stamp && nfast == 0) {                          // no frame went through render_r64_kernel: time the message with events
            j.stamp = e->stamped = false;
            CU(cudaEventRecord(e->ev0, e->stream));
        }
        if (q.chunk_frames > 0) {
            if (!k.render) return fail(e, SP_E_CUDA, "no render kernel linked for format %d", fmt);
            if ((rc = launch_render_kernel(e, k, j.plan, q))) return rc;
        }
    } else {
        // four-step path for n > 4096: radix-R pre-pass into a scratch, then the
        // 4096-point kernel in sub-frame mode, chunk by chunk
        const int R = j.plan.sub_r;
        const int n = p.n_full;
        const sp::Kernels &sub = kernels_for(SP_CF32);        // sub-frame input is always complex fp32
        if (!sub.render || !k.prepass) return fail(e, SP_E_CUDA, "no kernels linked for the four-step path");
        const float2 *twT = nullptr;
        int rc = get_table(e, Tw::big, n, &twT);
        if (rc) return rc;
        // frames per chunk: a 1 GB scratch (2^27 / n frames of n complex floats: a power of two, at least 512).  An L2-sized
        // scratch (<= 96 MB) keeps the 16 B/sample of scratch traffic out of HBM but leaves each launch with about one wave of
        // tiles; measured on B200 the large chunk wins (C5: 2.10 -> 1.56 ms, C3 x1: 1.28 -> 0.70 ms,
        // profiles/r01_fourstep_scratch_sweep.txt).
        long long ch = (1LL << 27) / n;
        if (ch > p.nframes) ch = (p.nframes + 7) / 8 * 8;
        if ((rc = ensure(e, e->scratch, (size_t)ch * (size_t)n * 8))) return rc;
        // split-real pairs bin k with bin n-k, which live in different sub-sequences: tap the whole spectrum of the
        // chunk and finish it in spectrum_epilogue_kernel
        const bool tap = p.channel_mode != 0;
        if (tap && (rc = ensure(e, e->spec, (size_t)ch * (size_t)n * 8))) return rc;
        const long long nf = p.nframes;
        sp::init_minmax_kernel<<<(unsigned)((nf + 255) / 256), 256, 0, e->stream>>>((unsigned *)p.fmin, (unsigned *)p.fmax, nf);
        e->launches++;
        long long big_done = 0;
        // Two forms of the four-step transform (measured side by side: profiles/r02_fourstep_paths.txt):
        //   ring  render_big_kernel: ONE persistent launch, the pre-pass output stays in an L2-resident ring - DRAM traffic 1.0 x the
        //         algorithmic bytes, but its pre-pass runs at one CTA per SM and is bound by the SM's load / store issue rate;
        //   hbm   prepass_kernel -> 1 GB scratch in HBM -> second-stage kernel: 2.3 x the traffic, a well-occupied pre-pass.
        // The ring form is as fast or faster where the scratch round trip hurts most - n = 32768 / 65536 on long captures (C3, C5) -
        // and slower elsewhere, so it is chosen there; SP_FOURSTEP=ring / hbm forces one form (tests, A/B runs).
        const char *force = getenv("SP_FOURSTEP");
        const bool force_hbm = force && !strcmp(force, "hbm"), force_ring = force && !strcmp(force, "ring");
        const bool ring = force_ring || (!force_hbm && (R == 8 || R == 16) && (double)nf * (double)n >= 536870912.0);
        if (fused == Route::fourstep && ring) {
            if ((rc = launch_big_kernel(e, k, p, &big_done))) return rc;
        } else release_l2_window(e);                          // the HBM-scratch form wants the whole cache
        for (long long c0 = big_done; c0 < nf; c0 += ch) {
            Params q = p;
            q.chunk_first = c0;
            q.chunk_frames = (nf - c0 < ch) ? nf - c0 : ch;
            CU(k.prepass(R, &q, (float2 *)e->scratch.p, twT, e->stream));
            q.sub_in = (const float2 *)e->scratch.p;
            e->launches++;
            Params full = q;                                   // what the epilogue kernel sees
            if (tap) { q.spec_out = (float2 *)e->spec.p; q.image = nullptr; q.db_out = nullptr; q.channel_mode = 0; }
            if (fused == Route::fourstep && sub.r64) {
                long long nfast = 0;
                if ((rc = launch_r64_kernel(e, sub, q, &nfast))) return rc;
                q.sub_in += (size_t)nfast * (size_t)R * 4096;
                q.chunk_first += nfast;
                q.chunk_frames -= nfast;
            }
            if (q.chunk_frames > 0 && (rc = launch_render_kernel(e, sub, j.plan, q))) return rc;
            if (tap) {
                const long long tiles = full.chunk_frames * (n / 256);
                const long long cap = (long long)e->sm_count * 8;
                sp::spectrum_epilogue_kernel<<<(unsigned)(tiles < cap ? tiles : cap), 256, (size_t)(sp::CB_RAW + full.cmap_len) * 4, e->stream>>>(
                    full, (const float2 *)e->spec.p);
                e->launches++;
            }
        }
    }
    return SP_OK;
}

// finalize_kernel, launched behind the render kernels with programmatic stream serialization: it starts while the render
// ends and, as it triggers before its wait, the next message's render_r64_kernel can start as soon as it is resident.  Its
// grid stays one CTA per 256 frames: capped at 8 or 32 CTAs it hid less of itself than it held back from the next render
// (C2 on B200: 0.2616 / 0.2483 against 0.2458 ms per step, profiles/r03_overlap_ab.txt).
static int enqueue_end(sp_engine *e, Job &j)
{
    Params &p = j.p;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((p.nframes + 255) / 256));
    cfg.blockDim = dim3(256);
    cfg.stream = e->stream;
    cfg.attrs = &attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    CU(cudaLaunchKernelEx(&cfg, sp::finalize_kernel,
        (const float *)p.fmin, (const float *)p.fmax, (const float2 *)p.fmid, p.nframes, j.range, j.gain, j.plan.sub_r > 1 ? 1 : 0,
        j.d_gmin, j.d_gmax, j.d_gamp, (unsigned *)e->mm.p, j.d_stats, (unsigned long long *)e->jhist.p, (const int2 *)e->jhtab.p,
        p.cmap_len, (unsigned long long *)e->acc.p, (unsigned long long *)e->acc.p + SP_CB_HIST_SIZE, j.d_cb, j.d_c,
        j.stamp ? (unsigned long long *)e->tstamp.p + 1 : (unsigned long long *)nullptr));
    e->launches++;
    e->acc_dirty = false;
    if (j.stamp) e->after_fin = true;
    else CU(cudaEventRecord(e->ev1, e->stream));
    return SP_OK;
}

static int enqueue(sp_engine *e, Job &j)
{
    int rc;
    if ((rc = enqueue_begin(e, j)) || (rc = enqueue_frames(e, j, j.p))) return rc;
    return enqueue_end(e, j);
}

static int finish(sp_engine *e, sp_reply *rp);

// ------------------------------------------------------------------ pipelined host-buffer path
// Host input -> host outputs for a long message: the frames are cut into chunks and three streams
// overlap the H2D copy of chunk i+1, the render of chunk i and the D2H copy of chunk i-1 (PCIe is
// full duplex), with two device buffers each for input bytes and image tiles.  Every chunk is a
// frame-range shard of the SAME message (global stride, global frame indices), so the result is
// bit-identical to the single-shot path; histograms accumulate across chunks, min / max / gauges
// are finalised once.  Host memory should be page-locked (sp_host_alloc_pinned) for real overlap.
// Frames per chunk of a message that takes this path, 0 for one that does not.
static long long pipeline_chunk_frames(const sp_request *rq)
{
    if ((rq->flags & (SP_F_BUFFER_ON_DEVICE | SP_F_REPLY_ON_DEVICE)) || rq->width <= 0 || rq->n <= 0 || rq->byte_length == 0) return 0;
    const char *env = getenv("SP_PIPE_MB");                  // chunk size in MB; 0 disables the pipeline
    const long long mb = env ? atoll(env) : 16;     // 16 MB: best of 8..128 on B200 + PCIe 5 (profiles/r01_e2e_chunk_sweep.txt)
    if (mb <= 0) return 0;
    const double in_per_frame = (double)rq->byte_length / (double)rq->width;
    const double out_per_frame = 4.0 * rq->n;
    const double per = in_per_frame > out_per_frame ? in_per_frame : out_per_frame;
    long long ch = (long long)((double)(mb << 20) / per);
    ch = ch / 8 * 8;
    if (ch < 64) ch = 64;
    return (rq->width >= 3 * ch) ? ch : 0;       // short messages: single shot
}

// Enqueue the copies of job j's five small reply arrays (gauges, histograms) to the non-null arrays of dst, in host memory.
static int copy_reply(sp_engine *e, const Job &j, const sp_reply &dst)
{
    const size_t W = (size_t)j.width;
    if (dst.gauge_mins) CU(cudaMemcpyAsync(dst.gauge_mins, j.d_gmin, W, cudaMemcpyDeviceToHost, e->stream));
    if (dst.gauge_maxs) CU(cudaMemcpyAsync(dst.gauge_maxs, j.d_gmax, W, cudaMemcpyDeviceToHost, e->stream));
    if (dst.gauge_amps) CU(cudaMemcpyAsync(dst.gauge_amps, j.d_gamp, W, cudaMemcpyDeviceToHost, e->stream));
    if (dst.cB_hist) CU(cudaMemcpyAsync(dst.cB_hist, j.d_cb, 8 * SP_CB_HIST_SIZE, cudaMemcpyDeviceToHost, e->stream));
    if (dst.c_hist) CU(cudaMemcpyAsync(dst.c_hist, j.d_c, 8 * (size_t)j.p.cmap_len, cudaMemcpyDeviceToHost, e->stream));
    return SP_OK;
}

// Byte offsets in sp_render_async's pinned bounce buffer for a message of W frames: [16 stats][W mins][W maxs][W amps], padded to
// 16 bytes, then [8 * SP_CB_HIST_SIZE cB][8 * cmap_len c], room for SP_MAX_CMAP colours.
struct Bounce {
    size_t gmin, gmax, gamp, cb, c, bytes;
    explicit Bounce(long long W)
        : gmin(16), gmax(16 + (size_t)W), gamp(16 + 2 * (size_t)W), cb(16 + (3 * (size_t)W + 15) / 16 * 16), c(cb + 8 * SP_CB_HIST_SIZE),
          bytes(c + 8 * (size_t)SP_MAX_CMAP) {}
};

static int render_pipelined(sp_engine *e, const sp_request *rq, sp_reply *rp, Job &j, long long ch, const Placement *pl,
                            sp_engine::Inflight *slot = nullptr)
{
    const int n = rq->n, sw = sp::sample_width(rq->format);
    const long long W = rq->width;
    const bool shard = rq->total_width != 0 || rq->total_byte_length != 0;
    const long long g_first = shard ? rq->frame_first : 0;                 // global index of local frame 0
    const long long buf_first = shard ? (long long)rq->buffer_first_sample : 0;
    const double stride = j.p.stride;
    if (!e->s_h2d) {
        CU(cudaStreamCreateWithFlags(&e->s_h2d, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&e->s_d2h, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CU(cudaEventCreateWithFlags(&e->ev_in[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&e->ev_comp[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&e->ev_out[i], cudaEventDisableTiming));
        }
        CU(cudaEventCreateWithFlags(&e->ev_setup, cudaEventDisableTiming));
    }
    int rc;
    // worst-case chunk input: ch frames at the global stride plus the window-length halo
    const size_t in_cap = (size_t)(((double)ch * stride + 2.0 * n + 64) * sw) + 64;
    const size_t img_cap = (size_t)4 * (size_t)ch * (size_t)n;
    for (int i = 0; i < 2; i++)
        if ((rc = ensure(e, e->pin[i], in_cap)) || (rc = ensure(e, e->pimg[i], img_cap))) return rc;
    if ((rc = enqueue_begin(e, j))) return rc;
    CU(cudaEventRecord(e->ev_setup, e->stream));                           // tables / window / LUT uploaded, histograms zeroed
    CU(cudaStreamWaitEvent(e->s_h2d, e->ev_setup, 0));
    CU(cudaStreamWaitEvent(e->s_d2h, e->ev_setup, 0));
    const long long nchunks = (W + ch - 1) / ch;
    for (long long c = 0; c < nchunks; c++) {
        const int b = (int)(c & 1);
        const long long x0 = c * ch, cw = (W - x0 < ch) ? W - x0 : ch;
        const bool msg_last = c == nchunks - 1 && (!shard || g_first + W == rq->total_width);
        const Span span = frame_span(stride, n, sw, g_first + x0, cw, buf_first, rq->byte_length, msg_last);
        const size_t bytes = span.b1 - span.b0;
        if (bytes + 16 > in_cap) return fail(e, SP_E_RANGE, "internal: pipeline chunk larger than its buffer");
        // input buffer b is free once the render of its previous user is done (chunk c-2, or a chunk of the previous message:
        // sp_render_async keeps two messages in flight)
        if (c >= 2 || e->pipe_used[b]) CU(cudaStreamWaitEvent(e->s_h2d, e->ev_comp[b], 0));
        CU(cudaMemcpyAsync(e->pin[b].p, (const uint8_t *)rq->buffer + span.b0, bytes, cudaMemcpyHostToDevice, e->s_h2d));
        CU(cudaEventRecord(e->ev_in[b], e->s_h2d));
        // render: needs the input, and image tile b drained by the D2H of chunk c-2
        CU(cudaStreamWaitEvent(e->stream, e->ev_in[b], 0));
        if ((c >= 2 || e->pipe_used[b]) && e->ev_out_valid[b]) CU(cudaStreamWaitEvent(e->stream, e->ev_out[b], 0));
        Params q = j.p;
        q.buf = (const uint8_t *)e->pin[b].p;
        q.valid_bytes = bytes;
        q.sample_base = span.s0;
        q.frame_first = g_first + x0;
        q.nframes = cw;
        q.chunk_first = 0;
        q.chunk_frames = cw;
        q.fmin = j.p.fmin + x0; q.fmax = j.p.fmax + x0; q.fmid = j.p.fmid + x0;
        q.image = j.d_image ? (uint8_t *)e->pimg[b].p : nullptr;
        if ((rc = enqueue_frames(e, j, q))) return rc;
        CU(cudaEventRecord(e->ev_comp[b], e->stream));
        if (j.d_image) {
            CU(cudaStreamWaitEvent(e->s_d2h, e->ev_comp[b], 0));
            if (rq->waterfall)      // rows [W - x0 - cw, W - x0) of the [W][n] image (lib/worker.js:116)
                CU(cudaMemcpyAsync(rp->image + (size_t)4 * n * (size_t)(W - x0 - cw), e->pimg[b].p, (size_t)4 * n * cw,
                                   cudaMemcpyDeviceToHost, e->s_d2h));
            else                    // columns [x0, x0 + cw) of the [n][W] image (lib/worker.js:117)
                CU(cudaMemcpy2DAsync(rp->image + 4 * (x0 + (pl ? pl->col0 : 0)), (size_t)4 * (pl ? pl->pitch_frames : W), e->pimg[b].p,
                                     (size_t)4 * cw, (size_t)4 * cw, (size_t)n, cudaMemcpyDeviceToHost, e->s_d2h));
            CU(cudaEventRecord(e->ev_out[b], e->s_d2h));
            e->ev_out_valid[b] = true;
        }
        e->pipe_used[b] = true;
    }
    if ((rc = enqueue_end(e, j))) return rc;
    if (slot) {
        // asynchronous form: the small reply arrays go through the slot's pinned bounce buffer (the caller's arrays may be pageable,
        // which would make the copies synchronous); the message is complete when they and the last image tiles have arrived
        uint8_t *b = slot->bounce;
        const Bounce at(W);
        sp_reply dst = {};
        dst.gauge_mins = b + at.gmin; dst.gauge_maxs = b + at.gmax; dst.gauge_amps = b + at.gamp;
        dst.cB_hist = (uint64_t *)(b + at.cb); dst.c_hist = (uint64_t *)(b + at.c);
        CU(cudaMemcpyAsync(b, e->stats_src, 16, cudaMemcpyDeviceToHost, e->stream));
        if ((rc = copy_reply(e, j, dst))) return rc;
        CU(cudaEventRecord(slot->reply, e->stream));
        CU(cudaStreamWaitEvent(e->s_done, slot->reply, 0));
        for (int i = 0; i < 2; i++)
            if (j.d_image && e->ev_out_valid[i]) CU(cudaStreamWaitEvent(e->s_done, e->ev_out[i], 0));
        CU(cudaEventRecord(slot->done, e->s_done));
        slot->launches = e->launches;
        return SP_OK;
    }
    if ((rc = copy_reply(e, j, *rp))) return rc;
    CU(cudaStreamSynchronize(e->s_d2h));
    return finish(e, rp);
}

static int finish(sp_engine *e, sp_reply *rp)
{
    double st[2];
    unsigned long long ts[2] = { 0, 0 };
    CU(cudaMemcpyAsync(st, e->stats_src, 16, cudaMemcpyDeviceToHost, e->stream));
    if (e->stamped) CU(cudaMemcpyAsync(ts, e->tstamp.p, 16, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    rp->dBfs_min = st[0];
    rp->dBfs_max = st[1];
    float ms = 0;
    if (e->stamped) ms = (float)((double)(long long)(ts[1] - ts[0]) * 1e-6);
    else CU(cudaEventElapsedTime(&ms, e->ev0, e->ev1));
    rp->device_ms = ms;
    rp->kernel_launches = e->launches;
    return SP_OK;
}

extern "C" int sp_render_enqueue(sp_engine *e, const sp_request *rq, sp_reply *rp)
{
    if (!e || !rq || !rp) return fail(e, SP_E_INVAL, "null argument");
    if (!e->subs.empty()) return fail(e, SP_E_INVAL, "sp_render_enqueue works on ONE device's buffers: use sp_render_shards on a multi-device engine");
    if (!(rq->flags & SP_F_BUFFER_ON_DEVICE) || !(rq->flags & SP_F_REPLY_ON_DEVICE))
        return fail(e, SP_E_INVAL, "sp_render_enqueue needs SP_F_BUFFER_ON_DEVICE | SP_F_REPLY_ON_DEVICE");
    Job j;
    int rc = prepare(e, rq, rp, j, false, nullptr);
    if (rc) return rc;
    if ((rc = enqueue(e, j))) return rc;
    e->pending = true;
    return SP_OK;
}

extern "C" int sp_render_finish(sp_engine *e, sp_reply *rp)
{
    e = dev0(e);
    if (!e || !rp) return fail(e, SP_E_INVAL, "null argument");
    if (!e->pending) return fail(e, SP_E_INVAL, "no render enqueued");
    e->pending = false;
    CU(cudaSetDevice(e->dev));
    return finish(e, rp);
}


// Device-resident shards of ONE message on a multi-device engine (lib/spectroplot.js:1206-1238 across GPUs, no host copy
// of anything): shard g lives on device g (its bytes, its image band, its gauges, its two histograms and a double[2] for
// min / max, all device pointers), the frame-range fields say which frames of the whole message it renders.  Every device
// renders its shard on its own stream; then ONE grouped NCCL all-reduce per device merges the histograms (sum, u64) and
// dBfs_min / dBfs_max (min / max, f64) in place over NVLink, so that every reply holds the statistics of the whole message.
extern "C" int sp_render_shards(sp_engine *e, const sp_request *rqs, sp_reply *rps)
{
    if (!e || !rqs || !rps) return fail(e, SP_E_INVAL, "null argument");
    if (e->subs.empty()) return fail(e, SP_E_INVAL, "sp_render_shards needs a multi-device engine (sp_create with ndev > 1)");
    NcclApi *nc = nccl_api();
    if (e->comms.empty()) return fail(e, SP_E_NCCL, "NCCL is not available: %s", e->nccl_err.c_str());
    const int G = (int)e->subs.size();
    for (int g = 0; g < G; g++) {
        const sp_request &rq = rqs[g];
        if (!(rq.flags & SP_F_BUFFER_ON_DEVICE) || !(rq.flags & SP_F_REPLY_ON_DEVICE))
            return fail(e, SP_E_INVAL, "shard %d: sp_render_shards needs SP_F_BUFFER_ON_DEVICE | SP_F_REPLY_ON_DEVICE", g);
        if (!rps[g].cB_hist || !rps[g].c_hist || !rps[g].minmax_dev)
            return fail(e, SP_E_INVAL, "shard %d: cB_hist, c_hist and minmax_dev (device pointers) are the merge targets", g);
        if (rq.cmap_len != rqs[0].cmap_len || rq.total_width != rqs[0].total_width || rq.total_width == 0)
            return fail(e, SP_E_RANGE, "shard %d: the shards must describe the same message (total_width, cmap_len)", g);
    }
    for (int g = 0; g < G; g++) {
        const int rc = sp_render_enqueue(e->subs[(size_t)g], &rqs[g], &rps[g]);
        if (rc) {
            e->err = "device " + std::to_string(e->subs[(size_t)g]->dev) + ": " + e->subs[(size_t)g]->err;
            for (int k = 0; k < g; k++) { cudaSetDevice(e->subs[(size_t)k]->dev); cudaStreamSynchronize(e->subs[(size_t)k]->stream); e->subs[(size_t)k]->pending = false; }
            return rc;
        }
    }
    int r = nc->GroupStart();
    for (int g = 0; g < G && r == 0; g++) {
        sp_engine *s = e->subs[(size_t)g];
        cudaSetDevice(s->dev);
        if (r == 0) r = nc->AllReduce(rps[g].cB_hist, rps[g].cB_hist, SP_CB_HIST_SIZE, SP_NCCL_UINT64, SP_NCCL_SUM, e->comms[(size_t)g], s->stream);
        if (r == 0) r = nc->AllReduce(rps[g].c_hist, rps[g].c_hist, (size_t)rqs[g].cmap_len, SP_NCCL_UINT64, SP_NCCL_SUM, e->comms[(size_t)g], s->stream);
        if (r == 0) r = nc->AllReduce(rps[g].minmax_dev, rps[g].minmax_dev, 1, SP_NCCL_FLOAT64, SP_NCCL_MIN, e->comms[(size_t)g], s->stream);
        if (r == 0) r = nc->AllReduce(rps[g].minmax_dev + 1, rps[g].minmax_dev + 1, 1, SP_NCCL_FLOAT64, SP_NCCL_MAX, e->comms[(size_t)g], s->stream);
    }
    const int r2 = nc->GroupEnd();
    if (r == 0) r = r2;
    int rc_out = SP_OK;
    for (int g = 0; g < G; g++) {            // wait for render + merge on every device; dBfs_min / max of the WHOLE message
        sp_engine *s = e->subs[(size_t)g];
        s->pending = false;
        cudaSetDevice(s->dev);
        const int rc = finish(s, &rps[g]);
        if (rc && !rc_out) { rc_out = rc; e->err = "device " + std::to_string(s->dev) + ": " + s->err; }
    }
    if (r != 0) return fail(e, SP_E_NCCL, "NCCL merge failed: %s", nc->GetErrorString ? nc->GetErrorString(r) : "error");
    return rc_out;
}

static int render_one(sp_engine *e, const sp_request *rq, sp_reply *rp, const Placement *pl)
{
    Job j;
    const long long ch = pipeline_chunk_frames(rq);
    j.pipelined = ch > 0;
    int rc = prepare(e, rq, rp, j, false, nullptr);
    if (rc) return rc;
    if (j.pipelined) return render_pipelined(e, rq, rp, j, ch, pl);
    if ((rc = enqueue(e, j))) return rc;
    const size_t W = (size_t)rq->width;
    if (!(rq->flags & SP_F_REPLY_ON_DEVICE)) {
        if (j.d_image) {
            if (pl && !rq->waterfall)       // a column band of the caller's [n][pitch] picture
                CU(cudaMemcpy2DAsync(rp->image + 4 * pl->col0, (size_t)4 * pl->pitch_frames, j.d_image, 4 * W, 4 * W, (size_t)rq->n,
                                     cudaMemcpyDeviceToHost, e->stream));
            else
                CU(cudaMemcpyAsync(rp->image, j.d_image, 4 * W * (size_t)rq->n, cudaMemcpyDeviceToHost, e->stream));
        }
        if ((rc = copy_reply(e, j, *rp))) return rc;
    }
    return finish(e, rp);
}

// ------------------------------------------------------------------ multi-device engine (sp_create with ndev > 1)
// One whole message, host buffers in and out: the frames are cut into ndev contiguous ranges on multiples of 8 frames
// (spectro_b200/sharding.py::plan_shards is the same plan), every device renders its range at the GLOBAL frame
// positions from its byte range plus an n-sample halo - one host thread per device, each running the ordinary
// single-device path (pipelined H2D / render / D2H) - and writes its column band (spectrogram) or row block
// (waterfall) straight into the caller's picture.  The only exchange is the merge of the two histograms and min / max
// (lib/spectroplot.js:1229-1238): ndev x ~10 KB, folded on the host.  (One process per GPU merges the same data with
// one NCCL all-gather instead: bench.py, spectro_b200/sharding.py.)
static int render_multi(sp_engine *e, const sp_request *rq, sp_reply *rp)
{
    if (rq->flags & (SP_F_BUFFER_ON_DEVICE | SP_F_REPLY_ON_DEVICE))
        return fail(e, SP_E_INVAL, "a multi-device engine takes host buffers (a device buffer lives on one GPU)");
    if (rq->total_width != 0 || rq->total_byte_length != 0)
        return fail(e, SP_E_INVAL, "a multi-device engine shards whole messages itself: leave the shard fields zero");
    const int G = (int)e->subs.size();
    const int sw = (rq->format >= 0 && rq->format < SP_FORMAT_COUNT) ? sp::sample_width(rq->format) : 0;
    const long long W = rq->width, n = rq->n;
    auto delegate = [&]() {                  // too small to split, or invalid: the first device alone (same checks, same errors)
        const int rc = render_one(e->subs[0], rq, rp, nullptr);
        if (rc) e->err = e->subs[0]->err;
        return rc;
    };
    if (sw <= 0 || n < SP_MIN_N || W < 16LL * G || !rq->buffer || (double)rq->byte_length / sw < (double)n) return delegate();
    const double sc = (double)rq->byte_length / (double)sw;
    const double stride = (sc - (double)n) / (double)(W - 1);                      // lib/worker.js:50, global
    auto cut = [&](int g) { return g >= G ? W : (g * W / G) / 8 * 8; };
    struct Part { sp_request rq; sp_reply rp; Placement pl; std::vector<uint64_t> cb, c; int rc = 0; bool used = false; };
    std::vector<Part> parts((size_t)G);
    int last_used = -1;
    for (int g = 0; g < G; g++) if (cut(g + 1) > cut(g)) last_used = g;
    for (int g = 0; g < G; g++) {
        const long long x0 = cut(g), x1 = cut(g + 1);
        if (x1 <= x0) continue;
        Part &pt = parts[(size_t)g];
        pt.used = true;
        const Span span = frame_span(stride, (int)n, sw, x0, x1 - x0, 0, rq->byte_length, g == last_used);
        pt.rq = *rq;
        pt.rq.buffer = (const uint8_t *)rq->buffer + span.b0;
        pt.rq.byte_length = span.b1 - span.b0;
        pt.rq.width = x1 - x0;
        pt.rq.total_byte_length = rq->byte_length;
        pt.rq.total_width = W;
        pt.rq.frame_first = x0;
        pt.rq.buffer_first_sample = (uint64_t)span.s0;
        memset(&pt.rp, 0, sizeof pt.rp);
        pt.pl = Placement{ W, x0 };
        if (rp->image) pt.rp.image = rq->waterfall ? rp->image + (size_t)4 * n * (size_t)(W - x1) : rp->image;   // rows [W - x1, W - x0)
        if (rp->gauge_mins) pt.rp.gauge_mins = rp->gauge_mins + x0;
        if (rp->gauge_maxs) pt.rp.gauge_maxs = rp->gauge_maxs + x0;
        if (rp->gauge_amps) pt.rp.gauge_amps = rp->gauge_amps + x0;
        pt.cb.assign(SP_CB_HIST_SIZE, 0);
        pt.c.assign((size_t)(rq->cmap_len > 0 ? rq->cmap_len : 1), 0);
        pt.rp.cB_hist = pt.cb.data();
        pt.rp.c_hist = pt.c.data();
    }
    std::vector<std::thread> threads;
    for (int g = 0; g < G; g++)
        if (parts[(size_t)g].used)
            threads.emplace_back([&, g]() { Part &pt = parts[(size_t)g]; pt.rc = render_one(e->subs[(size_t)g], &pt.rq, &pt.rp, &pt.pl); });
    for (auto &t : threads) t.join();
    for (int g = 0; g < G; g++)
        if (parts[(size_t)g].used && parts[(size_t)g].rc) {
            e->err = "device " + std::to_string(e->subs[(size_t)g]->dev) + ": " + e->subs[(size_t)g]->err;
            return parts[(size_t)g].rc;
        }
    // merge (lib/spectroplot.js:1229-1238): histograms add, min / max fold from the worker's initial values
    if (rp->cB_hist) memset(rp->cB_hist, 0, 8 * SP_CB_HIST_SIZE);
    if (rp->c_hist) memset(rp->c_hist, 0, 8 * (size_t)rq->cmap_len);
    rp->dBfs_min = 0.0;
    rp->dBfs_max = -200.0;
    rp->device_ms = 0.0f;
    rp->kernel_launches = 0;
    for (int g = 0; g < G; g++) {
        const Part &pt = parts[(size_t)g];
        if (!pt.used) continue;
        if (rp->cB_hist) for (int i = 0; i < SP_CB_HIST_SIZE; i++) rp->cB_hist[i] += pt.cb[(size_t)i];
        if (rp->c_hist) for (int i = 0; i < rq->cmap_len; i++) rp->c_hist[i] += pt.c[(size_t)i];
        if (pt.rp.dBfs_min < rp->dBfs_min) rp->dBfs_min = pt.rp.dBfs_min;
        if (pt.rp.dBfs_max > rp->dBfs_max) rp->dBfs_max = pt.rp.dBfs_max;
        if (pt.rp.device_ms > rp->device_ms) rp->device_ms = pt.rp.device_ms;
        rp->kernel_launches += pt.rp.kernel_launches;
    }
    return SP_OK;
}

extern "C" int sp_render(sp_engine *e, const sp_request *rq, sp_reply *rp)
{
    if (!e || !rq || !rp) return fail(e, SP_E_INVAL, "null argument");
    if (!e->subs.empty()) return render_multi(e, rq, rp);
    return render_one(e, rq, rp, nullptr);
}

// ---- asynchronous host-buffer messages (the reference posts messages to several workers and collects the replies as they come,
// lib/spectroplot.js:1206-1238; here two messages may be in flight on ONE engine so that the copy-out tail of a message
// overlaps the copy-in head of the next).  The reply struct and every buffer it points to must stay alive until sp_render_wait.
static int wait_slot(sp_engine *e, sp_engine::Inflight &s)
{
    if (!s.busy) return SP_OK;
    CU(cudaEventSynchronize(s.done));
    sp_reply *rp = s.rp;
    const size_t W = (size_t)s.width;
    const uint8_t *b = s.bounce;
    const Bounce at(s.width);
    double st[2];
    memcpy(st, b, 16);
    rp->dBfs_min = st[0];
    rp->dBfs_max = st[1];
    if (rp->gauge_mins) memcpy(rp->gauge_mins, b + at.gmin, W);
    if (rp->gauge_maxs) memcpy(rp->gauge_maxs, b + at.gmax, W);
    if (rp->gauge_amps) memcpy(rp->gauge_amps, b + at.gamp, W);
    if (rp->cB_hist) memcpy(rp->cB_hist, b + at.cb, 8 * SP_CB_HIST_SIZE);
    if (rp->c_hist) memcpy(rp->c_hist, b + at.c, 8 * (size_t)s.cmap_len);
    rp->device_ms = 0.0;                      // (per-message device time is not tracked for overlapping messages)
    rp->kernel_launches = s.launches;
    s.busy = false;
    return SP_OK;
}

extern "C" int sp_render_async(sp_engine *e, const sp_request *rq, sp_reply *rp, int *ticket)
{
    if (!e || !rq || !rp || !ticket) return fail(e, SP_E_INVAL, "null argument");
    if (!e->subs.empty()) return fail(e, SP_E_INVAL, "sp_render_async works on a single-device engine");
    CU(cudaSetDevice(e->dev));
    sp_engine::Inflight &s = e->inflight[e->next_ticket & 1];
    int rc = wait_slot(e, s);                              // at most two messages in flight: the older one is collected first
    if (rc) return rc;
    *ticket = e->next_ticket;
    s.ticket = e->next_ticket++;
    const long long ch = pipeline_chunk_frames(rq);
    if (ch <= 0) return render_one(e, rq, rp, nullptr);    // short or device-resident message: nothing to overlap, done on return
    if (!s.done) {
        CU(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&s.reply, cudaEventDisableTiming));
    }
    if (!e->s_done) CU(cudaStreamCreateWithFlags(&e->s_done, cudaStreamNonBlocking));
    const size_t need = Bounce(rq->width).bytes;
    if (s.bounce_cap < need) {
        if (s.bounce) cudaFreeHost(s.bounce);
        s.bounce = nullptr; s.bounce_cap = 0;
        CU(cudaHostAlloc((void **)&s.bounce, need, cudaHostAllocDefault));
        s.bounce_cap = need;
    }
    Job j;
    j.pipelined = true;
    if ((rc = prepare(e, rq, rp, j, false, nullptr))) return rc;
    if ((rc = render_pipelined(e, rq, rp, j, ch, nullptr, &s))) return rc;
    s.rp = rp;
    s.width = rq->width;
    s.cmap_len = rq->cmap_len;
    s.busy = true;
    return SP_OK;
}

extern "C" int sp_render_wait(sp_engine *e, int ticket)
{
    if (!e) return SP_E_INVAL;
    if (!e->subs.empty()) return fail(e, SP_E_INVAL, "sp_render_async works on a single-device engine");
    if (ticket < 0 || ticket >= e->next_ticket) return fail(e, SP_E_INVAL, "unknown ticket %d", ticket);
    sp_engine::Inflight &s = e->inflight[ticket & 1];
    if (s.ticket != ticket) return SP_OK;                  // already collected (by a later sp_render_async that needed the slot)
    CU(cudaSetDevice(e->dev));
    return wait_slot(e, s);
}

extern "C" int sp_render_zooms(sp_engine *e, const sp_request *rq, int nlevels, const int64_t *widths, sp_reply *replies)
{
    if (!e || !rq || !widths || !replies || nlevels < 1) return fail(e, SP_E_INVAL, "null argument or nlevels < 1");
    if (!rq->buffer) return fail(e, SP_E_INVAL, "buffer is required");
    sp_request r = *rq;
    int rc;
    if (!e->subs.empty()) {                                // every level is sharded across the devices like a single message
        for (int i = 0; i < nlevels; i++) {
            r.width = widths[i];
            if ((rc = sp_render(e, &r, &replies[i]))) return rc;
        }
        return SP_OK;
    }
    if (!(rq->flags & SP_F_BUFFER_ON_DEVICE)) {            // one upload shared by every level
        CU(cudaSetDevice(e->dev));
        if ((rc = ensure(e, e->zin, rq->byte_length + 16))) return rc;
        CU(cudaMemcpyAsync(e->zin.p, rq->buffer, rq->byte_length, cudaMemcpyHostToDevice, e->stream));
        r.buffer = e->zin.p;
        r.flags |= SP_F_BUFFER_ON_DEVICE;
    }
    for (int i = 0; i < nlevels; i++) {
        r.width = widths[i];
        if ((rc = sp_render(e, &r, &replies[i]))) return rc;
    }
    return SP_OK;
}

extern "C" int sp_render_db(sp_engine *e, const sp_request *rq, float *db)
{
    e = dev0(e);
    if (!e || !rq || !db) return fail(e, SP_E_INVAL, "null argument");
    const size_t cnt = (size_t)rq->width * (size_t)rq->n;
    int rc = ensure(e, e->db, cnt * 4);
    if (rc) return rc;
    sp_reply rp;
    memset(&rp, 0, sizeof rp);
    sp_request r2 = *rq;
    r2.flags &= ~SP_F_REPLY_ON_DEVICE;
    Job j;
    if ((rc = prepare(e, &r2, &rp, j, true, (float *)e->db.p))) return rc;
    if ((rc = enqueue(e, j))) return rc;
    CU(cudaMemcpyAsync(db, e->db.p, cnt * 4, cudaMemcpyDeviceToHost, e->stream));
    return finish(e, &rp);
}

extern "C" int sp_decode(sp_engine *e, int format, const void *bytes, uint64_t nbytes, uint64_t first, uint64_t count, float *iq)
{
    e = dev0(e);
    if (!e || !bytes || !iq) return fail(e, SP_E_INVAL, "null argument");
    if (format < 0 || format >= SP_FORMAT_COUNT) return fail(e, SP_E_BAD_FORMAT, "format %d out of range", format);
    if (count == 0) return SP_OK;
    CU(cudaSetDevice(e->dev));
    int rc;
    if ((rc = ensure(e, e->in, nbytes + 16)) || (rc = ensure(e, e->db, count * 8))) return rc;
    CU(cudaMemcpyAsync(e->in.p, bytes, nbytes, cudaMemcpyHostToDevice, e->stream));
    sp::decode_kernel<<<(unsigned)((count + 255) / 256), 256, 0, e->stream>>>((const uint8_t *)e->in.p, nbytes, format,
                                                                             (long long)first, (long long)count, (float2 *)e->db.p);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(iq, e->db.p, count * 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return SP_OK;
}

// ------------------------------------------------------------------ per-launch profiling ring
extern "C" int sp_profile_enable(sp_engine *e, int slots)
{
    e = dev0(e);
    if (!e) return SP_E_INVAL;
    e->prof_every = 1;
    e->prof_seq = 0;
    CU(cudaSetDevice(e->dev));
    for (auto ev : e->prof0) cudaEventDestroy(ev);
    for (auto ev : e->prof1) cudaEventDestroy(ev);
    e->prof0.clear(); e->prof1.clear(); e->prof_count = 0;
    for (int i = 0; i < slots; i++) {
        cudaEvent_t a, b;
        CU(cudaEventCreate(&a)); CU(cudaEventCreate(&b));
        e->prof0.push_back(a); e->prof1.push_back(b);
    }
    return SP_OK;
}
extern "C" int sp_profile_sample(sp_engine *e, int every)
{
    e = dev0(e);
    if (!e || every < 1) return SP_E_INVAL;
    e->prof_every = every;
    e->prof_seq = 0;
    return SP_OK;
}
extern "C" int sp_profile_read(sp_engine *e, float *ms, int max)
{
    e = dev0(e);
    if (!e || !ms) return SP_E_INVAL;
    CU(cudaSetDevice(e->dev));
    CU(cudaStreamSynchronize(e->stream));
    const long long slots = (long long)e->prof0.size();
    long long have = e->prof_count < slots ? e->prof_count : slots;
    if (have > max) have = max;
    for (long long i = 0; i < have; i++) {
        const long long idx = (e->prof_count - have + i) % slots;
        CU(cudaEventElapsedTime(&ms[i], e->prof0[idx], e->prof1[idx]));
    }
    e->prof_count = 0;
    return (int)have;
}

// ------------------------------------------------------------------ memory helpers
extern "C" int sp_device_alloc(sp_engine *e, uint64_t nbytes, void **dptr)
{
    e = dev0(e);
    if (!e || !dptr) return SP_E_INVAL;
    CU(cudaSetDevice(e->dev));
    CU(cudaMalloc(dptr, (size_t)((nbytes + 255) & ~255ull) + 256));
    return SP_OK;
}
extern "C" int sp_device_free(sp_engine *e, void *dptr)
{
    e = dev0(e);
    if (!e) return SP_E_INVAL;
    CU(cudaSetDevice(e->dev));
    CU(cudaFree(dptr));
    return SP_OK;
}
extern "C" int sp_memcpy_h2d(sp_engine *e, void *dst, const void *src, uint64_t n)
{
    e = dev0(e);
    if (!e) return SP_E_INVAL;
    CU(cudaSetDevice(e->dev));
    CU(cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return SP_OK;
}
extern "C" int sp_memcpy_d2h(sp_engine *e, void *dst, const void *src, uint64_t n)
{
    e = dev0(e);
    if (!e) return SP_E_INVAL;
    CU(cudaSetDevice(e->dev));
    CU(cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return SP_OK;
}
extern "C" int sp_host_alloc_pinned(uint64_t n, void **hptr)
{
    if (!hptr) return SP_E_INVAL;
    return cudaMallocHost(hptr, n) == cudaSuccess ? SP_OK : SP_E_CUDA;
}
extern "C" int sp_host_free_pinned(void *hptr) { return cudaFreeHost(hptr) == cudaSuccess ? SP_OK : SP_E_CUDA; }
extern "C" int sp_device_sync(sp_engine *e)
{
    if (!e) return SP_E_INVAL;
    if (!e->subs.empty()) {
        for (sp_engine *sub : e->subs) { const int rc = sp_device_sync(sub); if (rc) return rc; }
        return SP_OK;
    }
    CU(cudaSetDevice(e->dev));
    CU(cudaStreamSynchronize(e->stream));
    return SP_OK;
}

// ------------------------------------------------------------------ synthetic capture
extern "C" void sp_synth_lut(int16_t *lut)
{
    for (int j = 0; j < 4096; j++) lut[j] = (int16_t)lround(32767.0 * sin(2.0 * M_PI * j / 4096.0));
}

extern "C" int sp_synth_fill(sp_engine *e, void *dst_dev, int format, uint64_t first, uint64_t count, uint64_t total_samples, uint64_t seed)
{
    e = dev0(e);
    if (!e || !dst_dev) return fail(e, SP_E_INVAL, "null argument");
    if (format < 0 || format >= SP_FORMAT_COUNT) return fail(e, SP_E_BAD_FORMAT, "format %d out of range", format);
    CU(cudaSetDevice(e->dev));
    if (!e->synth_lut.p) {
        int rc = ensure(e, e->synth_lut, 8192);
        if (rc) return rc;
        int16_t lut[4096];
        sp_synth_lut(lut);
        CU(cudaMemcpyAsync(e->synth_lut.p, lut, 8192, cudaMemcpyHostToDevice, e->stream));
        CU(cudaStreamSynchronize(e->stream));
    }
    if (count == 0) return SP_OK;
    unsigned long long blocks = (count + 255) / 256;
    const unsigned long long cap = (unsigned long long)e->sm_count * 16;
    if (blocks > cap) blocks = cap;
    sp::synth_kernel<<<(unsigned)blocks, 256, 0, e->stream>>>((uint8_t *)dst_dev, format, first, count, total_samples, seed,
                                                              (const short *)e->synth_lut.p);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(e->stream));
    return SP_OK;
}
