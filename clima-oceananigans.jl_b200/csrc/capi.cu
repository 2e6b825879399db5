// capi.cu -- C ABI (include/ocean_b200.h), handles and the host-side orchestration of the
// NonhydrostaticModel time step.  No torch types, no CPU fallback.
#include "../../include/ocean_b200.h"
#include "internal.h"
#include "tma_util.cuh"

#include <algorithm>
#include <atomic>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

namespace ob {
namespace comm { bool peer_halo_error(); }
static thread_local std::string g_err;
static std::atomic<long long> g_launches{0};
static cudaStream_t g_stream = nullptr;
static cudaStream_t g_h2d = nullptr, g_d2h = nullptr;     // copy streams of the asynchronous parent transfers
static bool g_inited = false;

void count_launch(int n) { g_launches += n; }
static cudaStream_t g_override = nullptr;     // set while independent launches are spread over the side streams
cudaStream_t stream() { return g_override ? g_override : g_stream; }

static void ensure_device() {
    if (g_inited) return;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        throw Error(std::string("no usable CUDA device (libocean_b200 has no CPU fallback): ") +
                    (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    g_inited = true;
}

// ---- optional per-phase timing with CUDA events on the library stream (bench evidence) ----
struct Phase {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    double total_ms = 0;
    long long count = 0;
};
static bool g_profile = false;
static std::map<std::string, Phase> g_phases;
static std::vector<cudaEvent_t> g_event_pool;
static cudaEvent_t get_event() {
    if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
    cudaEvent_t e;
    OB_CUDA(cudaEventCreate(&e));
    return e;
}
struct ScopedPhase {
    Phase* ph = nullptr;
    cudaEvent_t a, b;
    cudaStream_t st = nullptr;
    explicit ScopedPhase(const char* name) {
        if (!g_profile) return;
        ph = &g_phases[name];
        a = get_event(); b = get_event();
        st = stream();
        cudaEventRecord(a, st);
    }
    ~ScopedPhase() {
        if (!ph) return;
        cudaEventRecord(b, st);
        ph->pending.emplace_back(a, b);
    }
};
PhaseScope::PhaseScope(const char* name) : impl(g_profile ? new ScopedPhase(name) : nullptr) {}
PhaseScope::~PhaseScope() { delete static_cast<ScopedPhase*>(impl); }
static void resolve_phases() {
    cudaStreamSynchronize(g_stream);
    for (auto& kv : g_phases) {
        for (auto& pr : kv.second.pending) {
            float ms = 0;
            cudaEventElapsedTime(&ms, pr.first, pr.second);
            kv.second.total_ms += ms;
            kv.second.count += 1;
            g_event_pool.push_back(pr.first);
            g_event_pool.push_back(pr.second);
        }
        kv.second.pending.clear();
    }
}
}  // namespace ob

using namespace ob;

#define API_BEGIN try {
#define API_END                                              \
    return 0;                                                \
    }                                                        \
    catch (const std::exception& e) {                        \
        ob::g_err = e.what();                                \
        return 1;                                            \
    }                                                        \
    catch (...) {                                            \
        ob::g_err = "unknown error";                         \
        return 2;                                            \
    }

// ---------------------------------------------------------------------------------------------
// handle types
// ---------------------------------------------------------------------------------------------
struct ob200_grid {
    int ftype;
    ob200_grid_desc desc;                   // host copy (pointers cleared)
    GridD<float> g32;
    GridD<double> g64;
    std::vector<void*> owned;
    std::vector<double> dzF_h, dzC_h;       // Julia indices 0..Nz+1 (for the tridiagonal solver)
    ~ob200_grid() { for (void* p : owned) cudaFree(p); }
};

struct ob200_field {
    const ob200_grid* grid;
    int loc[3];
    ob200_bc bcs[6];
    void* base = nullptr;                   // current buffer
    void* alt = nullptr;                    // second buffer (prognostic fields of a model)
    bool owns = true;
    int psize[3];
    void* staging = nullptr;                // device copy in the reference's parent layout (uploads)
    void* staging_out = nullptr;            // ... and a second one for asynchronous downloads
    void* bcv[6] = {};                      // array condition per side (ob200_field_set_boundary_values), null = bcs[s].value
    cudaEvent_t ev_in_ready = nullptr, ev_in_free = nullptr, ev_out_ready = nullptr, ev_out_free = nullptr;
    ~ob200_field() {
        for (void* p : bcv) if (p) cudaFree(p);
        if (owns) {
            // tensor maps over these buffers (tendency kernels) must not outlive them: the allocator may hand the same
            // address to a field of another grid
            const size_t bytes = grid ? (size_t)(grid->ftype == OB200_F32 ? grid->g32.total * 4 : grid->g64.total * 8) : 0;
            if (base) { ob::tmau::evict_maps(base, bytes); cudaFree(base); }
            if (alt) { ob::tmau::evict_maps(alt, bytes); cudaFree(alt); }
        }
        if (staging) cudaFree(staging);
        if (staging_out) cudaFree(staging_out);
        for (cudaEvent_t e : {ev_in_ready, ev_in_free, ev_out_ready, ev_out_free}) if (e) cudaEventDestroy(e);
    }
    template <class FT> FT* p0() const {
        return (FT*)base + (grid->ftype == OB200_F32 ? grid->g32.off0 : grid->g64.off0);
    }
    template <class FT> FT* alt0() const {
        return (FT*)alt + (grid->ftype == OB200_F32 ? grid->g32.off0 : grid->g64.off0);
    }
};

struct ob200_poisson {
    const ob200_grid* grid;
    int kind;
    PoissonPlan<float>* p32 = nullptr;
    PoissonPlan<double>* p64 = nullptr;
    ~ob200_poisson() { poisson_plan_destroy(p32); poisson_plan_destroy(p64); }
};

template <class FT> static const GridD<FT>& gridD(const ob200_grid* g);
template <> const GridD<float>& gridD<float>(const ob200_grid* g) { return g->g32; }
template <> const GridD<double>& gridD<double>(const ob200_grid* g) { return g->g64; }
template <class FT> static PoissonPlan<FT>* planOf(ob200_poisson* s);
template <> PoissonPlan<float>* planOf<float>(ob200_poisson* s) { return s->p32; }
template <> PoissonPlan<double>* planOf<double>(ob200_poisson* s) { return s->p64; }

static size_t fsize(const ob200_grid* g) { return g->ftype == OB200_F32 ? 4 : 8; }
static size_t gtotal(const ob200_grid* g) { return (size_t)(g->ftype == OB200_F32 ? g->g32.total : g->g64.total); }

// ---------------------------------------------------------------------------------------------
// library / memory
// ---------------------------------------------------------------------------------------------
extern "C" int32_t ob200_version(void) { return OB200_VERSION; }

extern "C" int32_t ob200_init(int32_t device) {
    API_BEGIN
    ensure_device();
    OB_CUDA(cudaSetDevice(device));
    OB_CUDA(cudaFree(0));
    API_END
}
extern "C" int32_t ob200_set_stream(void* s) { ob::g_stream = (cudaStream_t)s; return 0; }
extern "C" int32_t ob200_sync(void) {
    API_BEGIN
    ensure_device();
    OB_CUDA(cudaStreamSynchronize(stream()));
    if (ob::g_h2d) OB_CUDA(cudaStreamSynchronize(ob::g_h2d));
    if (ob::g_d2h) OB_CUDA(cudaStreamSynchronize(ob::g_d2h));
    if (ob::comm::peer_halo_error()) throw ob::Error("halo exchange: a neighbour's boundary planes did not arrive (peer-memory flag wait timed out)");
    API_END
}
// blocks until every download (ob200_field_get_parent_async) enqueued so far EXCEPT those of the most recent
// `keep_in_flight` ob200_mark_download_batch() batches has been delivered to host memory
static std::vector<cudaEvent_t> g_batch_events;
extern "C" int32_t ob200_mark_download_batch(void) {
    API_BEGIN
    if (!ob::g_d2h) return 0;
    cudaEvent_t e;
    OB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    OB_CUDA(cudaEventRecord(e, ob::g_d2h));
    g_batch_events.push_back(e);
    API_END
}
extern "C" int32_t ob200_sync_downloads(int32_t keep_in_flight) {
    API_BEGIN
    while ((int)g_batch_events.size() > std::max(0, keep_in_flight)) {
        cudaEvent_t e = g_batch_events.front();
        OB_CUDA(cudaEventSynchronize(e));
        cudaEventDestroy(e);
        g_batch_events.erase(g_batch_events.begin());
    }
    API_END
}
extern "C" size_t ob200_last_error(char* buf, size_t len) {
    size_t n = ob::g_err.size();
    if (buf && len) {
        size_t m = std::min(n, len - 1);
        memcpy(buf, ob::g_err.data(), m);
        buf[m] = 0;
    }
    return n;
}
extern "C" int64_t ob200_launch_count(void) { return ob::g_launches.load(); }

extern "C" int32_t ob200_malloc(void** p, size_t bytes) {
    API_BEGIN
    ensure_device();
    OB_CUDA(cudaMalloc(p, std::max<size_t>(bytes, 1)));
    API_END
}
extern "C" int32_t ob200_free(void* p) { API_BEGIN OB_CUDA(cudaFree(p)); API_END }
extern "C" int32_t ob200_memset(void* p, int32_t v, size_t bytes) {
    API_BEGIN OB_CUDA(cudaMemsetAsync(p, v, bytes, stream())); API_END
}
extern "C" int32_t ob200_upload(void* dst, const void* src, size_t bytes) {
    API_BEGIN
    OB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream()));
    OB_CUDA(cudaStreamSynchronize(stream()));
    API_END
}
extern "C" int32_t ob200_download(void* dst, const void* src, size_t bytes) {
    API_BEGIN
    OB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream()));
    OB_CUDA(cudaStreamSynchronize(stream()));
    API_END
}

// ---------------------------------------------------------------------------------------------
// grid
// ---------------------------------------------------------------------------------------------
template <class FT>
static void build_gridD(ob200_grid* G, GridD<FT>& g) {
    const ob200_grid_desc& D = G->desc;
    int align = sizeof(FT) == 8 ? 4 : 8;       // 32-byte sectors
    for (int d = 0; d < 3; ++d) {
        g.N[d] = D.N[d]; g.H[d] = D.H[d]; g.topo[d] = D.topology[d];
        g.regular[d] = D.regular[d];
        g.L[d] = (FT)D.L[d];
        g.d[d] = (FT)D.delta[d];
        g.dC[d] = g.dF[d] = nullptr;
        g.izC = g.izF = nullptr;
        if (D.topology[d] == OB200_FLAT) {
            if (D.N[d] != 1 || D.H[d] != 0) throw Error("Flat dimensions must have N = 1 and H = 0");
            g.O[d] = 0; g.S[d] = 1; g.regular[d] = 1; g.d[d] = 1; g.L[d] = 1;
        } else {
            if (D.N[d] < 1 || D.H[d] < 1) throw Error("non-Flat dimensions need N >= 1 and H >= 1");
            g.O[d] = d == 0 ? ((D.H[d] + align - 1) / align) * align : D.H[d];
            g.S[d] = g.O[d] + D.N[d] + D.H[d] + 1;
            if (d == 0) g.S[d] = ((g.S[d] + align - 1) / align) * align;
        }
    }
    for (int d = 0; d < 3; ++d) g.invd[d] = g.regular[d] ? FT(1) / g.d[d] : FT(0);
    g.st[0] = 1; g.st[1] = g.S[0]; g.st[2] = (long long)g.S[0] * g.S[1];
    g.total = (long long)g.S[0] * g.S[1] * g.S[2];
    g.off0 = (g.O[0] - 1) * g.st[0] + (g.O[1] - 1) * g.st[1] + (g.O[2] - 1) * g.st[2];
}

template <class FT>
static void upload_metrics(ob200_grid* G, GridD<FT>& g, const ob200_grid_desc* src) {
    if (g.regular[2] && g.topo[2] == OB_BOUNDED) {
        // constant reciprocal spacings in the table form the Bounded-z fused tendency kernel reads (tendency_fused.cu)
        const int lo = -g.H[2] - 1, hi = g.N[2] + g.H[2] + 2;
        std::vector<FT> v(hi - lo + 1, FT(1) / g.d[2]);
        FT* iptr = nullptr;
        OB_CUDA(cudaMalloc(&iptr, v.size() * sizeof(FT)));
        OB_CUDA(cudaMemcpy(iptr, v.data(), v.size() * sizeof(FT), cudaMemcpyHostToDevice));
        G->owned.push_back(iptr);
        g.izC = g.izF = iptr - lo;
    }
    for (int d = 0; d < 3; ++d) {
        if (g.regular[d]) continue;
        for (int w = 0; w < 2; ++w) {
            const double* h = w == 0 ? src->dC[d] : src->dF[d];
            int first = w == 0 ? src->dC_first[d] : src->dF_first[d];
            int len = w == 0 ? src->dC_len[d] : src->dF_len[d];
            if (!h || len <= 0) throw Error("stretched dimension without metric vectors");
            // need indices 1-H .. N+H for centers, 1-H .. N+H+1 for faces (when Bounded); clamp-extend
            int lo = std::min(first, -g.H[d] - 1), hi = std::max(first + len - 1, g.N[d] + g.H[d] + 2);
            std::vector<FT> v(hi - lo + 1);
            for (int q = lo; q <= hi; ++q) {
                int c = std::min(std::max(q, first), first + len - 1);
                v[q - lo] = (FT)h[c - first];
            }
            FT* dptr = nullptr;
            OB_CUDA(cudaMalloc(&dptr, v.size() * sizeof(FT)));
            OB_CUDA(cudaMemcpy(dptr, v.data(), v.size() * sizeof(FT), cudaMemcpyHostToDevice));
            G->owned.push_back(dptr);
            (w == 0 ? g.dC[d] : g.dF[d]) = dptr - lo;
            if (d == 2) {
                for (auto& x : v) x = FT(1) / x;
                FT* iptr = nullptr;
                OB_CUDA(cudaMalloc(&iptr, v.size() * sizeof(FT)));
                OB_CUDA(cudaMemcpy(iptr, v.data(), v.size() * sizeof(FT), cudaMemcpyHostToDevice));
                G->owned.push_back(iptr);
                (w == 0 ? g.izC : g.izF) = iptr - lo;
            }
        }
    }
}

extern "C" int32_t ob200_grid_create(const ob200_grid_desc* desc, ob200_grid** out) {
    API_BEGIN
    ensure_device();
    if (!desc || !out) throw Error("null argument");
    if (desc->ftype != OB200_F32 && desc->ftype != OB200_F64) throw Error("ftype must be OB200_F32 or OB200_F64");
    auto G = std::make_unique<ob200_grid>();
    G->ftype = desc->ftype;
    G->desc = *desc;
    build_gridD(G.get(), G->g32);
    build_gridD(G.get(), G->g64);
    if (G->ftype == OB200_F32) upload_metrics(G.get(), G->g32, desc);
    else upload_metrics(G.get(), G->g64, desc);
    // vertical spacings on the host for the Fourier-tridiagonal solver (Julia indices 0..Nz+1)
    int Nz = desc->N[2];
    G->dzF_h.assign(Nz + 2, desc->delta[2]);
    G->dzC_h.assign(Nz + 2, desc->delta[2]);
    if (!desc->regular[2] && desc->topology[2] != OB200_FLAT) {
        for (int k = 0; k <= Nz + 1; ++k) {
            int cf = std::min(std::max(k, desc->dF_first[2]), desc->dF_first[2] + desc->dF_len[2] - 1);
            int cc = std::min(std::max(k, desc->dC_first[2]), desc->dC_first[2] + desc->dC_len[2] - 1);
            G->dzF_h[k] = desc->dF[2][cf - desc->dF_first[2]];
            G->dzC_h[k] = desc->dC[2][cc - desc->dC_first[2]];
        }
    }
    for (int d = 0; d < 3; ++d) { G->desc.dC[d] = nullptr; G->desc.dF[d] = nullptr; }
    *out = G.release();
    API_END
}
extern "C" int32_t ob200_grid_destroy(ob200_grid* g) { delete g; return 0; }

// ---------------------------------------------------------------------------------------------
// fields
// ---------------------------------------------------------------------------------------------
static void parent_size(const ob200_grid* g, const int loc[3], int ps[3]) {
    for (int d = 0; d < 3; ++d) {
        const ob200_grid_desc& D = g->desc;
        if (D.topology[d] == OB200_FLAT) ps[d] = D.N[d];
        else ps[d] = D.N[d] + 2 * D.H[d] + ((loc[d] == OB200_FACE && D.topology[d] == OB200_BOUNDED) ? 1 : 0);
    }
}

static ob200_field* make_field(const ob200_grid* g, const int32_t loc[3], const ob200_bc bcs[6], bool two) {
    auto f = std::make_unique<ob200_field>();
    f->grid = g;
    for (int d = 0; d < 3; ++d) f->loc[d] = loc[d];
    for (int s = 0; s < 6; ++s) {
        if (bcs) f->bcs[s] = bcs[s];
        else {     // defaults: field_boundary_conditions.jl:13-30
            int d = s / 2, t = g->desc.topology[d];
            f->bcs[s].value = 0;
            f->bcs[s].kind = (t == OB200_PERIODIC || t == OB200_FULLY_CONNECTED) ? OB200_BC_PERIODIC
                           : t == OB200_FLAT ? OB200_BC_NONE
                           : (loc[d] == OB200_CENTER ? OB200_BC_FLUX : OB200_BC_OPEN);
        }
    }
    parent_size(g, f->loc, f->psize);
    size_t bytes = gtotal(g) * fsize(g);
    OB_CUDA(cudaMalloc(&f->base, bytes));
    OB_CUDA(cudaMemsetAsync(f->base, 0, bytes, stream()));
    if (two) {
        OB_CUDA(cudaMalloc(&f->alt, bytes));
        OB_CUDA(cudaMemsetAsync(f->alt, 0, bytes, stream()));
    }
    return f.release();
}

extern "C" int32_t ob200_field_create(const ob200_grid* g, const int32_t loc[3], const ob200_bc bcs[6],
                                      ob200_field** out) {
    API_BEGIN
    if (!g || !loc || !out) throw Error("null argument");
    *out = make_field(g, loc, bcs, false);
    API_END
}
extern "C" int32_t ob200_field_destroy(ob200_field* f) { delete f; return 0; }
extern "C" int32_t ob200_field_parent_size(const ob200_field* f, int32_t out[3]) {
    for (int d = 0; d < 3; ++d) out[d] = f->psize[d];
    return 0;
}

// Transfers of the reference's parent arrays.  The asynchronous variants run the DMA on two dedicated copy streams
// (one per direction: PCIe is full duplex) with their own staging buffers, ordered against the compute stream by
// events only, so that -- for a caller that streams host buffers through successive steps -- the upload of step
// n+1 and the download of step n overlap the kernels of the step in between.  ob200_sync() drains all three.
static void ensure_copy_streams() {
    if (!g_h2d) OB_CUDA(cudaStreamCreateWithFlags(&g_h2d, cudaStreamNonBlocking));
    if (!g_d2h) OB_CUDA(cudaStreamCreateWithFlags(&g_d2h, cudaStreamNonBlocking));
}
static void ensure_event(cudaEvent_t& e) {
    if (!e) OB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
}
template <class FT>
static void field_set_parent(ob200_field* f, const void* host, bool sync) {
    const GridD<FT>& g = gridD<FT>(f->grid);
    size_t n = (size_t)f->psize[0] * f->psize[1] * f->psize[2];
    if (!f->staging) OB_CUDA(cudaMalloc(&f->staging, n * sizeof(FT)));
    if (sync) {
        if (f->ev_in_free) OB_CUDA(cudaEventSynchronize(f->ev_in_free));
        OB_CUDA(cudaMemcpyAsync(f->staging, host, n * sizeof(FT), cudaMemcpyHostToDevice, stream()));
    } else {
        ensure_copy_streams();
        ensure_event(f->ev_in_ready);
        if (f->ev_in_free) OB_CUDA(cudaStreamWaitEvent(g_h2d, f->ev_in_free, 0));     // previous conversion has read the staging
        OB_CUDA(cudaMemcpyAsync(f->staging, host, n * sizeof(FT), cudaMemcpyHostToDevice, g_h2d));
        OB_CUDA(cudaEventRecord(f->ev_in_ready, g_h2d));
        OB_CUDA(cudaStreamWaitEvent(stream(), f->ev_in_ready, 0));
    }
    launch_to_internal<FT>(g, f->psize, f->loc, (const FT*)f->staging, (FT*)f->base);
    if (f->alt) launch_to_internal<FT>(g, f->psize, f->loc, (const FT*)f->staging, (FT*)f->alt);
    if (!sync) { ensure_event(f->ev_in_free); OB_CUDA(cudaEventRecord(f->ev_in_free, stream())); }
    if (sync) OB_CUDA(cudaStreamSynchronize(stream()));
}
template <class FT>
static void field_get_parent(ob200_field* f, void* host, bool sync) {
    const GridD<FT>& g = gridD<FT>(f->grid);
    size_t n = (size_t)f->psize[0] * f->psize[1] * f->psize[2];
    if (sync) {
        if (!f->staging) OB_CUDA(cudaMalloc(&f->staging, n * sizeof(FT)));
        if (f->ev_in_free) OB_CUDA(cudaEventSynchronize(f->ev_in_free));
        launch_from_internal<FT>(g, f->psize, f->loc, (const FT*)f->base, (FT*)f->staging);
        OB_CUDA(cudaMemcpyAsync(host, f->staging, n * sizeof(FT), cudaMemcpyDeviceToHost, stream()));
        OB_CUDA(cudaStreamSynchronize(stream()));
        return;
    }
    ensure_copy_streams();
    if (!f->staging_out) OB_CUDA(cudaMalloc(&f->staging_out, n * sizeof(FT)));
    ensure_event(f->ev_out_ready);
    if (f->ev_out_free) OB_CUDA(cudaStreamWaitEvent(stream(), f->ev_out_free, 0));     // previous DMA has drained the staging
    launch_from_internal<FT>(g, f->psize, f->loc, (const FT*)f->base, (FT*)f->staging_out);
    OB_CUDA(cudaEventRecord(f->ev_out_ready, stream()));
    OB_CUDA(cudaStreamWaitEvent(g_d2h, f->ev_out_ready, 0));
    OB_CUDA(cudaMemcpyAsync(host, f->staging_out, n * sizeof(FT), cudaMemcpyDeviceToHost, g_d2h));
    ensure_event(f->ev_out_free);
    OB_CUDA(cudaEventRecord(f->ev_out_free, g_d2h));
}
extern "C" int32_t ob200_field_set_parent(ob200_field* f, const void* host) {
    API_BEGIN
    if (f->grid->ftype == OB200_F32) field_set_parent<float>(f, host, true);
    else field_set_parent<double>(f, host, true);
    API_END
}
extern "C" int32_t ob200_field_get_parent(const ob200_field* f, void* host) {
    API_BEGIN
    if (f->grid->ftype == OB200_F32) field_get_parent<float>(const_cast<ob200_field*>(f), host, true);
    else field_get_parent<double>(const_cast<ob200_field*>(f), host, true);
    API_END
}
extern "C" int32_t ob200_field_set_parent_async(ob200_field* f, const void* host) {
    API_BEGIN
    if (f->grid->ftype == OB200_F32) field_set_parent<float>(f, host, false);
    else field_set_parent<double>(f, host, false);
    API_END
}
extern "C" int32_t ob200_field_get_parent_async(const ob200_field* f, void* host) {
    API_BEGIN
    if (f->grid->ftype == OB200_F32) field_get_parent<float>(const_cast<ob200_field*>(f), host, false);
    else field_get_parent<double>(const_cast<ob200_field*>(f), host, false);
    API_END
}
// ---- output path: the gather / reduction runs on the device into a stream-ordered temporary, the (small) result travels on
// the download stream like ob200_field_get_parent_async
static void interior_size(const ob200_field* f, int n[3]) {
    const ob200_grid_desc& D = f->grid->desc;
    for (int d = 0; d < 3; ++d)
        n[d] = D.N[d] + ((f->loc[d] == OB200_FACE && D.topology[d] == OB200_BOUNDED) ? 1 : 0);
}
template <class FT, class Launch>
static void device_result_to_host(size_t count, void* host, Launch&& launch) {
    if (count == 0) return;
    ensure_copy_streams();
    FT* tmp = nullptr;
    OB_CUDA(cudaMallocAsync(&tmp, count * sizeof(FT), stream()));
    launch(tmp);
    cudaEvent_t ready;
    OB_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    OB_CUDA(cudaEventRecord(ready, stream()));
    OB_CUDA(cudaStreamWaitEvent(g_d2h, ready, 0));
    OB_CUDA(cudaEventDestroy(ready));           // released once the recorded work has completed
    OB_CUDA(cudaMemcpyAsync(host, tmp, count * sizeof(FT), cudaMemcpyDeviceToHost, g_d2h));
    OB_CUDA(cudaFreeAsync(tmp, g_d2h));
}
template <class FT>
static void field_slice(const ob200_field* f, const int32_t lo[3], const int32_t hi[3], void* host) {
    const GridD<FT>& g = gridD<FT>(f->grid);
    const ob200_grid_desc& D = f->grid->desc;
    int ni[3], l[3], n[3];
    interior_size(f, ni);
    for (int d = 0; d < 3; ++d) {
        const int H = D.topology[d] == OB200_FLAT ? 0 : D.H[d];
        if (lo[d] < 1 - H || hi[d] > ni[d] + H || hi[d] < lo[d]) throw Error("field slice: index range outside the field (halos included)");
        l[d] = lo[d]; n[d] = hi[d] - lo[d] + 1;
    }
    const FT* p0 = f->template p0<FT>();
    device_result_to_host<FT>((size_t)n[0] * n[1] * n[2], host, [&](FT* tmp) { launch_slice<FT>(g, p0, l, n, tmp); });
}
template <class FT>
static void field_average(const ob200_field* f, const int32_t dims[3], void* host) {
    const GridD<FT>& g = gridD<FT>(f->grid);
    int n[3], a[3];
    interior_size(f, n);
    size_t outs = 1;
    for (int d = 0; d < 3; ++d) { a[d] = dims[d] != 0; outs *= a[d] ? 1 : (size_t)n[d]; }
    const FT* p0 = f->template p0<FT>();
    device_result_to_host<FT>(outs, host, [&](FT* tmp) { launch_average<FT>(g, p0, n, a, tmp); });
}
extern "C" int32_t ob200_field_slice_async(const ob200_field* f, const int32_t lo[3], const int32_t hi[3], void* host) {
    API_BEGIN
    if (!f || !lo || !hi || !host) throw Error("null argument");
    if (f->grid->ftype == OB200_F32) field_slice<float>(f, lo, hi, host);
    else field_slice<double>(f, lo, hi, host);
    API_END
}
extern "C" int32_t ob200_field_average_async(const ob200_field* f, const int32_t dims[3], void* host) {
    API_BEGIN
    if (!f || !dims || !host) throw Error("null argument");
    if (f->grid->ftype == OB200_F32) field_average<float>(f, dims, host);
    else field_average<double>(f, dims, host);
    API_END
}
extern "C" int32_t ob200_field_device_view(const ob200_field* f, void** base, int64_t off[1], int64_t st[3]) {
    const ob200_grid* G = f->grid;
    bool s = G->ftype == OB200_F32;
    *base = f->base;
    off[0] = s ? G->g32.off0 + G->g32.st[0] + G->g32.st[1] + G->g32.st[2]
               : G->g64.off0 + G->g64.st[0] + G->g64.st[1] + G->g64.st[2];
    for (int d = 0; d < 3; ++d) st[d] = s ? G->g32.st[d] : G->g64.st[d];
    return 0;
}

// entry q of a halo batch: field f with its boundary conditions (constant values and array tables)
template <class FT>
static void halo_entry(HaloBatch<FT>& hb, int q, const ob200_field* f) {
    hb.p0[q] = f->p0<FT>();
    for (int d = 0; d < 3; ++d) hb.loc[q][d] = f->loc[d];
    for (int s = 0; s < 6; ++s) {
        hb.bc_kind[q][s] = f->bcs[s].kind;
        hb.bc_val[q][s] = (FT)f->bcs[s].value;
        hb.bc_tab[q][s] = (const FT*)f->bcv[s];
    }
}
// the constant Flux boundary conditions the tendency kernels add themselves: a side with an array condition is "no constant
// flux" there, because the boundary-plane pass (model_boundary_fluxes) adds it
template <class FT>
static FluxBC<FT> constant_flux_bcs(const ob200_field* f) {
    FluxBC<FT> fbc;
    for (int s = 0; s < 6; ++s) { fbc.kind[s] = f->bcs[s].kind; fbc.val[s] = f->bcv[s] ? FT(0) : (FT)f->bcs[s].value; }
    return fbc;
}

template <class FT>
static void fill_halos(ob200_field* const* fields, int n) {
    if (n == 0) return;
    const ob200_grid* G = fields[0]->grid;
    const GridD<FT>& g = gridD<FT>(G);
    for (int start = 0; start < n; start += MAXF) {
        HaloBatch<FT> hb;
        hb.n = std::min(MAXF, n - start);
        for (int q = 0; q < hb.n; ++q) {
            ob200_field* f = fields[start + q];
            if (f->grid != G) throw Error("fill_halo_regions: fields live on different grids");
            halo_entry<FT>(hb, q, f);
        }
        launch_fill_halos<FT>(g, hb);
    }
}
extern "C" int32_t ob200_fill_halo_regions(ob200_field* const* fields, int32_t n) {
    API_BEGIN
    if (n <= 0) return 0;
    if (fields[0]->grid->ftype == OB200_F32) fill_halos<float>(fields, n);
    else fill_halos<double>(fields, n);
    API_END
}

// FluxBoundaryCondition(Q) / ValueBoundaryCondition(Q) / GradientBoundaryCondition(Q) with a 2-D array Q
// (BoundaryConditions/boundary_condition.jl: getbc(bc::BC{<:Any,<:AbstractArray}, i, j, grid, ...) = bc.condition[i, j])
extern "C" int32_t ob200_field_set_boundary_values(ob200_field* f, int32_t side, const void* values) {
    API_BEGIN
    if (!f) throw Error("null argument");
    if (side < 0 || side > 5) throw Error("boundary values: side out of range");
    static const char* names[6] = {"west", "east", "south", "north", "bottom", "top"};
    const std::string who = std::string("boundary values of the ") + names[side] + " side: ";
    const ob200_grid_desc& D = f->grid->desc;
    const int d = side / 2;
    for (int e = 0; e < 3; ++e)
        if (D.topology[e] == OB200_FULLY_CONNECTED)
            throw Error(who + "array conditions are not supported on a slab-decomposed (FullyConnected) grid");
    if (D.topology[d] != OB200_BOUNDED) throw Error(who + "the dimension is not Bounded (Periodic, Flat or FullyConnected)");
    const int kind = f->bcs[side].kind;
    if (kind != OB200_BC_FLUX && kind != OB200_BC_VALUE && kind != OB200_BC_GRADIENT)
        throw Error(who + "array conditions need a Flux, Value or Gradient boundary condition (not Open / None)");
    if (f->loc[d] == OB200_FACE)
        throw Error(who + "the field is located on the faces normal to this side (the impenetrable wall)");
    if (!values) {
        if (f->bcv[side]) {
            OB_CUDA(cudaStreamSynchronize(stream()));      // kernels enqueued so far may still read the table
            OB_CUDA(cudaFree(f->bcv[side]));
            f->bcv[side] = nullptr;
        }
        return 0;
    }
    size_t count = 1;
    for (int e = 0; e < 3; ++e)
        if (e != d) count *= (size_t)D.N[e];           // a Flat dimension has N = 1
    const size_t bytes = count * fsize(f->grid);
    if (!f->bcv[side]) OB_CUDA(cudaMalloc(&f->bcv[side], bytes));
    // on the library stream: after every step enqueued so far (a step joins its side streams before its last kernel), before
    // the next one.  A pageable source is staged before the call returns; a pinned one is read by the DMA itself, so wait for it
    OB_CUDA(cudaMemcpyAsync(f->bcv[side], values, bytes, cudaMemcpyHostToDevice, stream()));
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, values) != cudaSuccess) cudaGetLastError();    // the query's own error only
    else if (pa.type == cudaMemoryTypeHost) OB_CUDA(cudaStreamSynchronize(stream()));
    API_END
}

static double* g_red = nullptr;
static double* red_buf() {
    if (!g_red) OB_CUDA(cudaMalloc(&g_red, 8 * sizeof(double)));
    return g_red;
}
extern "C" int32_t ob200_field_reduce(const ob200_field* f, double* sum, double* sumsq, double* maxabs,
                                      int32_t* has_nan) {
    API_BEGIN
    int n[3];
    for (int d = 0; d < 3; ++d) {
        const ob200_grid_desc& D = f->grid->desc;
        n[d] = D.N[d] + ((f->loc[d] == OB200_FACE && D.topology[d] == OB200_BOUNDED) ? 1 : 0);
    }
    double* r = red_buf();
    if (f->grid->ftype == OB200_F32) launch_reduce<float>(f->grid->g32, f->p0<float>(), n, r);
    else launch_reduce<double>(f->grid->g64, f->p0<double>(), n, r);
    double h[4];
    OB_CUDA(cudaMemcpyAsync(h, r, sizeof(h), cudaMemcpyDeviceToHost, stream()));
    OB_CUDA(cudaStreamSynchronize(stream()));
    if (sum) *sum = h[0];
    if (sumsq) *sumsq = h[1];
    if (maxabs) *maxabs = h[2];
    if (has_nan) *has_nan = h[3] > 0;
    API_END
}

// ---------------------------------------------------------------------------------------------
// Poisson solvers
// ---------------------------------------------------------------------------------------------
static int pick_solver(const ob200_grid* g, int kind) {
    const ob200_grid_desc& D = g->desc;
    if (kind == OB200_SOLVER_AUTO)     // NonhydrostaticModels.jl:18-27
        kind = (D.regular[0] && D.regular[1] && D.regular[2]) ? OB200_SOLVER_FFT : OB200_SOLVER_FOURIER_TRIDIAGONAL;
    if (kind == OB200_SOLVER_FFT && !(D.regular[0] && D.regular[1] && D.regular[2]))
        throw Error("FFTBasedPoissonSolver requires a regular grid");
    if (kind == OB200_SOLVER_FOURIER_TRIDIAGONAL) {
        if (D.topology[2] != OB200_BOUNDED)
            throw Error("FourierTridiagonalPoissonSolver can only be used with a Bounded z topology.");
        if (!(D.regular[0] && D.regular[1])) throw Error("FourierTridiagonalPoissonSolver requires regular x and y");
    }
    return kind;
}
extern "C" int32_t ob200_poisson_create(const ob200_grid* g, int32_t kind, ob200_poisson** out) {
    API_BEGIN
    ensure_device();
    auto s = std::make_unique<ob200_poisson>();
    s->grid = g;
    s->kind = pick_solver(g, kind);
    if (g->ftype == OB200_F32) s->p32 = poisson_plan_create<float>(g->g32, s->kind, g->dzF_h.data(), g->dzC_h.data());
    else s->p64 = poisson_plan_create<double>(g->g64, s->kind, g->dzF_h.data(), g->dzC_h.data());
    *out = s.release();
    API_END
}
extern "C" int32_t ob200_poisson_destroy(ob200_poisson* s) { delete s; return 0; }

template <class FT> struct C2 { FT x, y; };

template <class FT>
static void poisson_solve_host(ob200_poisson* s, ob200_field* phi, const void* rhs_host) {
    const ob200_grid* G = s->grid;
    const GridD<FT>& g = gridD<FT>(G);
    PoissonPlan<FT>* p = planOf<FT>(s);
    if (rhs_host && poisson_has_fast<FT>(p)) {
        size_t n = (size_t)g.N[0] * g.N[1] * g.N[2];
        FT* tmp = nullptr;
        OB_CUDA(cudaMalloc(&tmp, n * sizeof(FT)));
        OB_CUDA(cudaMemcpyAsync(tmp, rhs_host, n * sizeof(FT), cudaMemcpyHostToDevice, stream()));
        poisson_solve_real<FT>(p, g, tmp, phi->p0<FT>());
        OB_CUDA(cudaStreamSynchronize(stream()));
        cudaFree(tmp);
        return;
    }
    if (rhs_host) {
        size_t n = (size_t)g.N[0] * g.N[1] * g.N[2];
        std::vector<C2<FT>> h(n);
        const FT* r = (const FT*)rhs_host;
        for (size_t q = 0; q < n; ++q) {
            FT v = r[q];
            if (s->kind == OB200_SOLVER_FOURIER_TRIDIAGONAL) {       // set_source_term!: times Δzᶜ
                int k = (int)(q / ((size_t)g.N[0] * g.N[1]));
                v = v * (FT)G->dzC_h[k + 1];
            }
            h[q].x = v; h[q].y = 0;
        }
        OB_CUDA(cudaMemcpyAsync(poisson_storage(p), h.data(), n * sizeof(C2<FT>), cudaMemcpyHostToDevice, stream()));
        OB_CUDA(cudaStreamSynchronize(stream()));
    }
    poisson_solve<FT>(p, g, phi->p0<FT>());
}
extern "C" int32_t ob200_poisson_solve(ob200_poisson* s, ob200_field* phi, const void* rhs_host) {
    API_BEGIN
    if (s->grid != phi->grid) throw Error("solver and field live on different grids");
    if (s->grid->ftype == OB200_F32) poisson_solve_host<float>(s, phi, rhs_host);
    else poisson_solve_host<double>(s, phi, rhs_host);
    API_END
}

template <class FT>
static void solve_for_pressure_T(ob200_poisson* s, ob200_field* p, double dt, const ob200_field* u,
                                 const ob200_field* v, const ob200_field* w) {
    using CT = typename std::conditional<sizeof(FT) == 4, float2, double2>::type;
    const GridD<FT>& g = gridD<FT>(s->grid);
    PoissonPlan<FT>* pl = planOf<FT>(s);
    if (poisson_has_fast<FT>(pl)) {
        poisson_solve_velocities<FT>(pl, g, u->p0<FT>(), v->p0<FT>(), w->p0<FT>(), (FT)dt, p->p0<FT>());
        return;
    }
    launch_pressure_rhs<FT, CT>(g, u->p0<FT>(), v->p0<FT>(), w->p0<FT>(), (FT)dt,
                                s->kind == OB200_SOLVER_FOURIER_TRIDIAGONAL, (CT*)poisson_storage(pl));
    poisson_solve<FT>(pl, g, p->p0<FT>());
}
extern "C" int32_t ob200_solve_for_pressure(ob200_poisson* s, ob200_field* p, double dt, const ob200_field* u,
                                            const ob200_field* v, const ob200_field* w) {
    API_BEGIN
    if (s->grid->ftype == OB200_F32) solve_for_pressure_T<float>(s, p, dt, u, v, w);
    else solve_for_pressure_T<double>(s, p, dt, u, v, w);
    API_END
}

template <class FT>
static void tridiag_host(int cplx, int Nx, int Ny, int Nz, const double* a, const double* b, const double* c,
                         const void* rhs, void* phi) {
    size_t n = (size_t)Nx * Ny * Nz, es = sizeof(FT) * (cplx ? 2 : 1);
    double *da, *db, *dc;
    void *dr, *dp;
    FT* dt;
    OB_CUDA(cudaMalloc(&da, std::max(1, Nz - 1) * sizeof(double)));
    OB_CUDA(cudaMalloc(&dc, std::max(1, Nz - 1) * sizeof(double)));
    OB_CUDA(cudaMalloc(&db, n * sizeof(double)));
    OB_CUDA(cudaMalloc(&dr, n * es));
    OB_CUDA(cudaMalloc(&dp, n * es));
    OB_CUDA(cudaMalloc(&dt, n * sizeof(FT)));
    OB_CUDA(cudaMemcpy(da, a, (Nz - 1) * sizeof(double), cudaMemcpyHostToDevice));
    OB_CUDA(cudaMemcpy(dc, c, (Nz - 1) * sizeof(double), cudaMemcpyHostToDevice));
    OB_CUDA(cudaMemcpy(db, b, n * sizeof(double), cudaMemcpyHostToDevice));
    OB_CUDA(cudaMemcpy(dr, rhs, n * es, cudaMemcpyHostToDevice));
    OB_CUDA(cudaMemset(dp, 0, n * es));
    OB_CUDA(cudaMemset(dt, 0, n * sizeof(FT)));
    batched_tridiagonal<FT>(Nx, Ny, Nz, cplx != 0, da, db, dc, dr, dp, dt);
    OB_CUDA(cudaStreamSynchronize(stream()));
    OB_CUDA(cudaMemcpy(phi, dp, n * es, cudaMemcpyDeviceToHost));
    cudaFree(da); cudaFree(db); cudaFree(dc); cudaFree(dr); cudaFree(dp); cudaFree(dt);
}
extern "C" int32_t ob200_batched_tridiagonal_solve(int32_t ftype, int32_t cplx, int32_t Nx, int32_t Ny, int32_t Nz,
                                                   const double* a, const double* b, const double* c,
                                                   const void* rhs, void* phi) {
    API_BEGIN
    ensure_device();
    if (ftype == OB200_F32) tridiag_host<float>(cplx, Nx, Ny, Nz, a, b, c, rhs, phi);
    else tridiag_host<double>(cplx, Nx, Ny, Nz, a, b, c, rhs, phi);
    API_END
}

// ---------------------------------------------------------------------------------------------
// model
// ---------------------------------------------------------------------------------------------
struct ob200_model {
    ob200_model_desc desc;
    const ob200_grid* grid;
    int nf;                                         // prognostic fields: 3 + ntracers
    std::vector<std::unique_ptr<ob200_field>> F;    // state (two buffers each)
    std::vector<std::unique_ptr<ob200_field>> Gn, Gm;
    std::unique_ptr<ob200_field> pNHS, pHY;
    std::unique_ptr<ob200_field> nue;               // SmagorinskyLilly / AMD eddy viscosity (diffusivity_fields.νₑ)
    std::vector<std::unique_ptr<ob200_field>> kappae;     // AMD eddy diffusivities (diffusivity_fields.κₑ), one per tracer
    std::unique_ptr<ob200_field> ivd_scratch;             // Thomas scratch of the vertically implicit diffusion step
    std::vector<std::unique_ptr<ob200_field>> bg;         // background_fields per prognostic field (null: none)
    std::unique_ptr<ob200_field> bg_zero;                 // the missing background velocities when another one is given
    std::unique_ptr<ob200_poisson> solver;
    std::vector<void*> owned;
    Phys<float> P32;
    Phys<double> P64;
    double time = 0, previous_dt = 1.0 / 0.0;
    long long iteration = 0;
    bool use_fast = true;
    // side streams / events of this model (independent launches of a stage are forked onto them and joined before the
    // stage's next dependent kernel); created on first use, released with the model
    cudaStream_t side[3] = {nullptr, nullptr, nullptr}, hy_stream = nullptr;
    // neighbour exchange of a stage in flight on its own stream while the next stage's interior tiles run (model_halo_*)
    cudaStream_t halo_stream = nullptr;
    cudaEvent_t ev_halo_a = nullptr, ev_halo_b = nullptr;
    bool halo_pending = false;
    cudaEvent_t ev_fork = nullptr, ev_join[3] = {nullptr, nullptr, nullptr}, hy_fork = nullptr, hy_done = nullptr;
    ~ob200_model() {
        for (void* p : owned) cudaFree(p);
        for (cudaStream_t s : {side[0], side[1], side[2], hy_stream, halo_stream}) if (s) cudaStreamDestroy(s);
        for (cudaEvent_t e : {ev_halo_a, ev_halo_b}) if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : {ev_fork, ev_join[0], ev_join[1], ev_join[2], hy_fork, hy_done}) if (e) cudaEventDestroy(e);
    }
};
template <class FT> static Phys<FT>& physOf(ob200_model* m);
template <> Phys<float>& physOf<float>(ob200_model* m) { return m->P32; }
template <> Phys<double>& physOf<double>(ob200_model* m) { return m->P64; }

// interior node count of prognostic field q (u, v, w: Face along q) along dimension d
static int forcing_table_length(const ob200_grid_desc& G, int q, int d) {
    return G.N[d] + ((q == d && G.topology[d] == OB200_BOUNDED) ? 1 : 0);
}

template <class FT>
static void build_phys(ob200_model* m) {
    Phys<FT>& P = physOf<FT>(m);
    const ob200_model_desc& D = m->desc;
    P.g = gridD<FT>(m->grid);
    P.scheme = D.advection;
    P.zweno = D.weno_zweno;
    static const int buf[7] = {0, 0, 1, 1, 1, 2, 2};
    P.buffer = buf[D.advection];
    for (int d = 0; d < 3; ++d)
        for (int l = 0; l < 2; ++l) {
            P.wc[d][l] = nullptr;
            if (d == 2) P.wzp[l] = nullptr;
            if (D.advection == OB200_ADV_WENO5 && D.weno_coeff[d][l]) {
                size_t n = 4 * (size_t)(P.g.N[d] + 2) * 3;
                std::vector<FT> h(n);
                for (size_t q = 0; q < n; ++q) h[q] = (FT)D.weno_coeff[d][l][q];
                FT* dp = nullptr;
                OB_CUDA(cudaMalloc(&dp, n * sizeof(FT)));
                OB_CUDA(cudaMemcpy(dp, h.data(), n * sizeof(FT), cudaMemcpyHostToDevice));
                m->owned.push_back(dp);
                P.wc[d][l] = dp;
                if (d == 2) {
                    // the same coefficients packed for tendency_fused.cu: entry (k, side) = 10 values at (2 k + side) * 10,
                    // side 1 = left-biased: 2 x the nine coefficients of the window ordered towards the face (the right-biased
                    // row is the natural one reversed), so both sides are one arithmetic on one 80-byte row
                    const int n2 = P.g.N[d] + 2;
                    std::vector<FT> pk((size_t)n2 * 2 * 10, FT(0));
                    for (int kk = 0; kk < n2; ++kk)
                        for (int j = 0; j < 9; ++j) {
                            const int mL = j / 3, cL = j % 3, jr = 8 - j, mR = jr / 3, cR = jr % 3;
                            pk[((size_t)2 * kk + 1) * 10 + j] = 2 * h[((size_t)(1 + mL) * n2 + kk) * 3 + cL];
                            pk[((size_t)2 * kk + 0) * 10 + j] = 2 * h[((size_t)(0 + mR) * n2 + kk) * 3 + cR];
                        }
                    FT* pp = nullptr;
                    OB_CUDA(cudaMalloc(&pp, pk.size() * sizeof(FT)));
                    OB_CUDA(cudaMemcpy(pp, pk.data(), pk.size() * sizeof(FT), cudaMemcpyHostToDevice));
                    m->owned.push_back(pp);
                    P.wzp[l] = pp;
                }
            }
        }
    if (D.advection == OB200_ADV_WENO5 && P.g.topo[2] == OB_BOUNDED && P.g.regular[2] && !P.wzp[0]) {
        // regular Bounded z: the uniform coefficients (weno_fifth_order.jl:518-524) in the same packed form; the window
        // ordered towards the face makes the two sides' rows identical
        const double cu[9] = {1.0 / 3, 5.0 / 6, -1.0 / 6, -1.0 / 6, 5.0 / 6, 1.0 / 3, 1.0 / 3, -7.0 / 6, 11.0 / 6};
        const int n2 = P.g.N[2] + 2;
        std::vector<FT> pk((size_t)n2 * 2 * 10, FT(0));
        for (int r = 0; r < 2 * n2; ++r)
            for (int j = 0; j < 9; ++j) pk[(size_t)r * 10 + j] = (FT)(2 * cu[j]);
        FT* pp = nullptr;
        OB_CUDA(cudaMalloc(&pp, pk.size() * sizeof(FT)));
        OB_CUDA(cudaMemcpy(pp, pk.data(), pk.size() * sizeof(FT), cudaMemcpyHostToDevice));
        m->owned.push_back(pp);
        P.wzp[0] = P.wzp[1] = pp;
    }
    P.closure = D.closure;
    P.vitd = D.closure_vertically_implicit;
    P.nu = (FT)D.nu;
    for (int t = 0; t < 8; ++t) P.kappa[t] = (FT)(D.closure == OB200_CLOSURE_SMAGORINSKY_LILLY ? D.prandtl[t] : D.kappa[t]);
    P.smagC = (FT)D.smagorinsky_C; P.smagCb = (FT)D.smagorinsky_Cb;
    P.nue = m->nue ? m->nue->template p0<FT>() : nullptr;
    P.amdCnu = (FT)D.amd_Cnu; P.amdCb = (FT)D.amd_Cb; P.amdHasCb = D.amd_has_Cb;
    for (int t = 0; t < 8; ++t) {
        P.amdCk[t] = (FT)D.amd_Ckappa[t];
        P.kappae[t] = t < (int)m->kappae.size() ? m->kappae[t]->template p0<FT>() : nullptr;
    }
    P.fplane = D.coriolis_fplane;
    P.f = (FT)D.f;
    P.btr = D.buoyancy_tracer;
    P.tilted = D.gravity_tilted;
    for (int d = 0; d < 3; ++d) P.ghat[d] = (FT)D.g_hat[d];
    P.ntr = D.ntracers;
    // Relaxation forcings: the host's tables rounded to FT, stored at index 1..n (Julia index) of a model-owned buffer
    auto table = [&](const double* src, int n) -> const FT* {
        std::vector<FT> h(n + 1, FT(0));
        for (int q = 0; q < n; ++q) h[q + 1] = (FT)src[q];
        FT* dp = nullptr;
        OB_CUDA(cudaMalloc(&dp, h.size() * sizeof(FT)));
        m->owned.push_back(dp);
        OB_CUDA(cudaMemcpy(dp, h.data(), h.size() * sizeof(FT), cudaMemcpyHostToDevice));
        return dp;
    };
    for (int q = 0; q < 3 + 8; ++q) {
        Relax<FT>& r = P.frc[q];
        r = Relax<FT>{0, -1, -1, nullptr, nullptr, FT(0), FT(0)};
        const ob200_forcing& F = D.forcing[q];
        if (q >= m->nf || !F.active) continue;
        r.on = 1;
        r.md = F.mask_dim; r.td = F.target_dim;
        r.mc = (FT)F.rate; r.tc = (FT)F.target_value;
        if (r.md >= 0) r.M = table(F.mask, forcing_table_length(m->grid->desc, q, r.md));
        if (r.td >= 0) r.T = table(F.target, forcing_table_length(m->grid->desc, q, r.td));
    }
    for (int q = 0; q < 3 + 8; ++q) P.bg[q] = q < m->nf && m->bg[q] ? m->bg[q]->template p0<FT>() : nullptr;
    for (int d = 0; d < 3; ++d) P.bgU[d] = P.bg[d] ? P.bg[d] : (m->bg_zero ? m->bg_zero->template p0<FT>() : nullptr);
}

extern "C" int32_t ob200_model_create(const ob200_model_desc* desc, ob200_model** out) {
    API_BEGIN
    ensure_device();
    if (!desc || !desc->grid || !out) throw Error("null argument");
    if (desc->ntracers < 0 || desc->ntracers > OB200_MAX_TRACERS) throw Error("too many tracers");
    if (desc->advection < 0 || desc->advection > OB200_ADV_WENO5) throw Error("unsupported advection scheme");
    if (desc->closure < 0 || desc->closure > OB200_CLOSURE_AMD) throw Error("unsupported closure");
    if (desc->closure_vertically_implicit) {
        // implicit_diffusion_solver (vertically_implicit_diffusion_solver.jl:95-108) + the supported set of this library
        if (desc->closure != OB200_CLOSURE_3D && desc->closure != OB200_CLOSURE_VERTICAL)
            throw Error("VerticallyImplicitTimeDiscretization is supported for ScalarDiffusivity (ThreeDimensional / Vertical) only");
        if (desc->grid->desc.topology[2] != OB200_BOUNDED)
            throw Error("VerticallyImplicitTimeDiscretization can only be specified on grids that are Bounded in the z-direction.");
    }
    if (desc->closure == OB200_CLOSURE_SMAGORINSKY_LILLY)
        for (int t = 0; t < desc->ntracers; ++t)
            if (!(desc->prandtl[t] > 0)) throw Error("SmagorinskyLilly needs a positive Prandtl number for every tracer");
    if (desc->buoyancy_tracer >= desc->ntracers) throw Error("buoyancy tracer index out of range");
    if (desc->buoyancy_kind < 0 || desc->buoyancy_kind > 1) throw Error("unsupported buoyancy model");
    if (desc->buoyancy_kind == 1) {
        if (desc->temperature_tracer >= desc->ntracers || desc->salinity_tracer >= desc->ntracers)
            throw Error("temperature / salinity tracer index out of range");
        if (desc->temperature_tracer < 0 && desc->salinity_tracer < 0)
            throw Error("SeawaterBuoyancy needs an active temperature or salinity tracer");
    }
    const ob200_grid_desc& GD = desc->grid->desc;
    // Relaxation forcings (Forcings/relaxation.jl): tables along non-Flat dimensions only, present where a dimension is given
    for (int q = 0; q < 3 + OB200_MAX_TRACERS; ++q) {
        const ob200_forcing& F = desc->forcing[q];
        if (!F.active) continue;
        const std::string who = "forcing of prognostic field " + std::to_string(q);
        if (q >= 3 + desc->ntracers) throw Error(who + ": the model has no such field");
        for (int pass = 0; pass < 2; ++pass) {
            const int d = pass ? F.target_dim : F.mask_dim;
            const double* t = pass ? F.target : F.mask;
            const char* what = pass ? "target" : "mask";
            if (d < -1 || d > 2) throw Error(who + ": " + what + " dimension out of range");
            if (d >= 0 && GD.topology[d] == OB200_FLAT) throw Error(who + ": " + what + " along a Flat dimension");
            if (d >= 0 && !t) throw Error(who + ": " + what + " table missing");
        }
    }
    // required halo: Advection.jl:40 (buffer + 1), closures need 1
    static const int need[7] = {1, 1, 2, 2, 2, 3, 3};
    for (int d = 0; d < 3; ++d)
        if (GD.topology[d] != OB200_FLAT && GD.H[d] < need[desc->advection])
            throw Error("grid halo too small for the advection scheme (the host shim must inflate it, "
                        "nonhydrostatic_model.jl:140-148)");
    auto m = std::make_unique<ob200_model>();
    m->desc = *desc;
    m->grid = desc->grid;
    m->nf = 3 + desc->ntracers;
    for (int q = 0; q < m->nf; ++q) {
        int32_t loc[3] = {OB200_CENTER, OB200_CENTER, OB200_CENTER};
        if (q < 3) loc[q] = OB200_FACE;
        m->F.emplace_back(make_field(m->grid, loc, desc->bcs[q], true));
        m->Gn.emplace_back(make_field(m->grid, loc, nullptr, false));
        m->Gm.emplace_back(make_field(m->grid, loc, nullptr, false));
    }
    int32_t ccc[3] = {0, 0, 0};
    m->pNHS.reset(make_field(m->grid, ccc, nullptr, false));
    if (GD.topology[2] != OB200_FLAT) m->pHY.reset(make_field(m->grid, ccc, nullptr, false));
    if (desc->closure == OB200_CLOSURE_SMAGORINSKY_LILLY || desc->closure == OB200_CLOSURE_AMD)
        m->nue.reset(make_field(m->grid, ccc, nullptr, false));
    if (desc->closure == OB200_CLOSURE_AMD)
        for (int t = 0; t < desc->ntracers; ++t) m->kappae.emplace_back(make_field(m->grid, ccc, nullptr, false));
    if (desc->closure_vertically_implicit) m->ivd_scratch.reset(make_field(m->grid, ccc, nullptr, false));
    // background_fields: model-owned copies of the host's parent arrays (halos included, never filled)
    m->bg.resize(m->nf);
    for (int q = 0; q < 3 + OB200_MAX_TRACERS; ++q) {
        if (!desc->background[q]) continue;
        if (q >= m->nf) throw Error("background of prognostic field " + std::to_string(q) + ": the model has no such field");
        int32_t loc[3] = {OB200_CENTER, OB200_CENTER, OB200_CENTER};
        if (q < 3) loc[q] = OB200_FACE;
        m->bg[q].reset(make_field(m->grid, loc, nullptr, false));
        if (m->grid->ftype == OB200_F32) field_set_parent<float>(m->bg[q].get(), desc->background[q], true);
        else field_set_parent<double>(m->bg[q].get(), desc->background[q], true);
    }
    if ((m->bg[0] || m->bg[1] || m->bg[2]) && !(m->bg[0] && m->bg[1] && m->bg[2]))
        m->bg_zero.reset(make_field(m->grid, ccc, nullptr, false));       // zeroed on creation
    ob200_poisson* s = nullptr;
    if (ob200_poisson_create(m->grid, desc->pressure_solver, &s)) throw Error(ob::g_err);
    m->solver.reset(s);
    if (m->grid->ftype == OB200_F32) build_phys<float>(m.get());
    else build_phys<double>(m.get());
    for (int d = 0; d < 3; ++d) for (int l = 0; l < 2; ++l) m->desc.weno_coeff[d][l] = nullptr;
    for (ob200_forcing& F : m->desc.forcing) F.mask = F.target = nullptr;      // borrowed host tables: copied to the device
    for (const void*& p : m->desc.background) p = nullptr;
    *out = m.release();
    if (ob200_model_update_state(*out)) { delete *out; *out = nullptr; throw Error(ob::g_err); }
    API_END
}
extern "C" int32_t ob200_model_destroy(ob200_model* m) { delete m; return 0; }

extern "C" int32_t ob200_model_field(ob200_model* m, const char* name, ob200_field** out) {
    API_BEGIN
    std::string s(name);
    auto idx = [&](const std::string& t) -> int {
        if (t == "u") return 0;
        if (t == "v") return 1;
        if (t == "w") return 2;
        if (t.size() >= 2 && t[0] == 'c') {
            int k = std::stoi(t.substr(1));
            if (k >= 0 && k < m->desc.ntracers) return 3 + k;
        }
        return -1;
    };
    ob200_field* f = nullptr;
    if (s == "pNHS") f = m->pNHS.get();
    else if (s == "nu_e") f = m->nue.get();
    else if (s.rfind("kappa_e", 0) == 0) { int k = std::stoi(s.substr(7)); if (k >= 0 && k < (int)m->kappae.size()) f = m->kappae[k].get(); }
    else if (s == "pHY") f = m->pHY.get();
    else if (s.rfind("Gn_", 0) == 0) { int q = idx(s.substr(3)); if (q >= 0) f = m->Gn[q].get(); }
    else if (s.rfind("Gm_", 0) == 0) { int q = idx(s.substr(3)); if (q >= 0) f = m->Gm[q].get(); }
    else if (s.rfind("bg_", 0) == 0) { int q = idx(s.substr(3)); if (q >= 0) f = m->bg[q].get(); }
    else { int q = idx(s); if (q >= 0) f = m->F[q].get(); }
    if (!f) throw Error("no such model field: " + s);
    *out = f;
    API_END
}

template <class FT>
static void model_fill_state_halos(ob200_model* m, int first, int last) {
    std::vector<ob200_field*> v;
    for (int q = first; q < last; ++q) v.push_back(m->F[q].get());
    fill_halos<FT>(v.data(), (int)v.size());
}

// the buoyancy model with the CURRENT state pointers (the state buffers swap every substep)
template <class FT>
static Buoy<FT> model_buoyancy(ob200_model* m) {
    const ob200_model_desc& D = m->desc;
    Buoy<FT> b{};
    b.mode = BUOY_NONE;
    auto tr = [&](int idx) -> const FT* { return m->F[3 + idx]->template p0<FT>(); };
    if (D.buoyancy_kind == 1) {
        b.g = (FT)D.gravitational_acceleration; b.alpha = (FT)D.thermal_expansion; b.beta = (FT)D.haline_contraction;
        b.ga = b.g * b.alpha; b.ngb = (-b.g) * b.beta;
        if (D.temperature_tracer >= 0 && D.salinity_tracer >= 0) { b.mode = BUOY_TS; b.T = tr(D.temperature_tracer); b.S = tr(D.salinity_tracer); }
        else if (D.temperature_tracer >= 0) { b.mode = BUOY_T; b.T = tr(D.temperature_tracer); }
        else if (D.salinity_tracer >= 0) { b.mode = BUOY_S; b.S = tr(D.salinity_tracer); }
    } else if (D.buoyancy_tracer >= 0) {
        b.mode = BUOY_TRACER; b.T = tr(D.buoyancy_tracer);
    }
    return b;
}

template <class FT>
static void model_hydrostatic(ob200_model* m, bool periodic_images) {
    ScopedPhase phase_timer("hydrostatic");
    const GridD<FT>& g = gridD<FT>(m->grid);
    Phys<FT>& P = physOf<FT>(m);
    const Buoy<FT> b = model_buoyancy<FT>(m);
    FT gz = (b.mode && P.tilted) ? P.ghat[2] : FT(1);
    launch_hydrostatic_pressure<FT>(g, b, gz, m->pHY->template p0<FT>(), periodic_images);
}

// calculate_diffusivities! + fill_halo_regions!(diffusivity_fields) (update_nonhydrostatic_model_state.jl:29-31): needs
// valid halos of the velocities and of the buoyancy tracers
template <class FT>
static void model_diffusivities(ob200_model* m) {
    if (!m->nue) return;
    ScopedPhase ph("closure");
    Phys<FT>& P = physOf<FT>(m);
    if (m->desc.closure == OB200_CLOSURE_AMD) {
        const FT* cs[8]; FT* ks[8];
        std::vector<ob200_field*> fl = {m->nue.get()};
        for (size_t t = 0; t < m->kappae.size(); ++t) {
            cs[t] = m->F[3 + t]->template p0<FT>(); ks[t] = m->kappae[t]->template p0<FT>();
            fl.push_back(m->kappae[t].get());
        }
        launch_amd<FT>(P, model_buoyancy<FT>(m), m->F[0]->template p0<FT>(), m->F[1]->template p0<FT>(),
                       m->F[2]->template p0<FT>(), m->nue->template p0<FT>(), (int)m->kappae.size(), cs, ks);
        fill_halos<FT>(fl.data(), (int)fl.size());
        return;
    }
    launch_smagorinsky<FT>(P, model_buoyancy<FT>(m), m->F[0]->template p0<FT>(), m->F[1]->template p0<FT>(),
                           m->F[2]->template p0<FT>(), m->nue->template p0<FT>());
    ob200_field* f = m->nue.get();
    fill_halos<FT>(&f, 1);
}

template <class FT>
static void model_update_state(ob200_model* m, bool tracers_too = true) {
    // update_nonhydrostatic_model_state.jl:14-37
    { ScopedPhase ph("halo"); model_fill_state_halos<FT>(m, 0, tracers_too ? m->nf : 3); }
    model_diffusivities<FT>(m);
    if (m->pHY) {
        model_hydrostatic<FT>(m, false);
        ScopedPhase ph("halo");
        ob200_field* ph_ = m->pHY.get();
        fill_halos<FT>(&ph_, 1);
    }
}
// fill_halos in two phases on two streams (slab-decomposed y, peer-memory exchange): the Periodic halos of the owned rows on the
// library stream, then the neighbour exchange + the Periodic halos of the received rows on the model's halo stream.  The next
// tendency launch runs its interior tiles meanwhile and calls model_halo_join before its boundary tiles
// (Distributed/halo_communication.jl:62-183 overlaps the same way with asynchronous MPI requests).
template <class FT>
static void fill_halos_overlapped(ob200_model* m, ob200_field* const* fields, int n) {
    const ob200_grid* G = fields[0]->grid;
    const GridD<FT>& g = gridD<FT>(G);
    if (!m->halo_stream) {
        OB_CUDA(cudaStreamCreateWithFlags(&m->halo_stream, cudaStreamNonBlocking));
        OB_CUDA(cudaEventCreateWithFlags(&m->ev_halo_a, cudaEventDisableTiming));
        OB_CUDA(cudaEventCreateWithFlags(&m->ev_halo_b, cudaEventDisableTiming));
    }
    auto batch = [&](int start) {
        HaloBatch<FT> hb;
        hb.n = std::min(MAXF, n - start);
        for (int q = 0; q < hb.n; ++q) halo_entry<FT>(hb, q, fields[start + q]);
        return hb;
    };
    for (int start = 0; start < n; start += MAXF) launch_fill_halos_phase<FT>(g, batch(start), 0);
    OB_CUDA(cudaEventRecord(m->ev_halo_a, g_stream));
    OB_CUDA(cudaStreamWaitEvent(m->halo_stream, m->ev_halo_a, 0));
    g_override = m->halo_stream;
    try {
        for (int start = 0; start < n; start += MAXF) launch_fill_halos_phase<FT>(g, batch(start), 1);
    } catch (...) { g_override = nullptr; throw; }
    g_override = nullptr;
    OB_CUDA(cudaEventRecord(m->ev_halo_b, m->halo_stream));
    m->halo_pending = true;
}
static void model_halo_join(ob200_model* m) {
    if (!m->halo_pending) return;
    OB_CUDA(cudaStreamWaitEvent(g_stream, m->ev_halo_b, 0));
    m->halo_pending = false;
}

// update_state! as it runs inside time_step!, after model_pressure_step(..., tracers_too = true): tracer halos are
// already valid, so pHY' is integrated first and velocities + pHY' share ONE halo fill (one neighbour exchange
// on the slab-decomposed path instead of two).  Same values as the reference sequence.
// fused (all non-Flat dimensions Periodic, see model_fused_periodic): the solver, the pressure correction and the
// hydrostatic integral read their operands with periodic wrap-around, so ALL halo fills of the stage (state
// before the solve, pNHS after it, state + pHY' here) collapse into this one single-launch shell fill.
template <class FT>
static void model_update_state_after_projection(ob200_model* m, bool fused, bool hydrostatic_done = false,
                                                bool overlap_next = false) {
    std::vector<ob200_field*> v = {m->F[0].get(), m->F[1].get(), m->F[2].get()};
    if (m->pHY) {
        if (!hydrostatic_done) model_hydrostatic<FT>(m, fused);
        v.push_back(m->pHY.get());
    }
    if (fused) {
        for (int q = 3; q < m->nf; ++q) v.push_back(m->F[q].get());
        v.push_back(m->pNHS.get());
    }
    static const bool no_overlap = getenv("OB200_NO_HALO_OVERLAP") != nullptr;
    if (overlap_next && fused && !no_overlap && !m->nue && m->use_fast && halo_overlap_supported<FT>(gridD<FT>(m->grid))) {
        ScopedPhase ph("halo");
        fill_halos_overlapped<FT>(m, v.data(), (int)v.size());
        return;
    }
    { ScopedPhase ph("halo"); fill_halos<FT>(v.data(), (int)v.size()); }
    model_diffusivities<FT>(m);
}
// Fused stage: the hydrostatic integral depends only on the buoyancy tracer, which is final once the tendency kernels
// have run, so it is enqueued on a side stream and overlaps the pressure solve and the correction (it is a
// latency-bound column walk that leaves most of the machine idle).  Returns true if it was started.
template <class FT>
static bool model_hydrostatic_async_begin(ob200_model* m) {
    if (!m->pHY) return false;
    if (!m->hy_stream) {
        OB_CUDA(cudaStreamCreateWithFlags(&m->hy_stream, cudaStreamNonBlocking));
        OB_CUDA(cudaEventCreateWithFlags(&m->hy_fork, cudaEventDisableTiming));
        OB_CUDA(cudaEventCreateWithFlags(&m->hy_done, cudaEventDisableTiming));
    }
    OB_CUDA(cudaEventRecord(m->hy_fork, g_stream));
    OB_CUDA(cudaStreamWaitEvent(m->hy_stream, m->hy_fork, 0));
    g_override = m->hy_stream;
    try { model_hydrostatic<FT>(m, true); } catch (...) { g_override = nullptr; throw; }
    g_override = nullptr;
    OB_CUDA(cudaEventRecord(m->hy_done, m->hy_stream));
    return true;
}
static void model_hydrostatic_async_end(ob200_model* m) { OB_CUDA(cudaStreamWaitEvent(g_stream, m->hy_done, 0)); }

// the fused path: every non-Flat dimension Periodic (not slab-decomposed) and regular, fast FFT solver
template <class FT>
static bool model_fused_periodic(ob200_model* m) {
    return periodic_wrap_supported<FT>(gridD<FT>(m->grid)) && poisson_has_fast<FT>(planOf<FT>(m->solver.get()));
}
extern "C" int32_t ob200_model_update_state(ob200_model* m) {
    API_BEGIN
    if (m->grid->ftype == OB200_F32) model_update_state<float>(m);
    else model_update_state<double>(m);
    API_END
}

// calculate_boundary_tendency_contributions! of the array Flux conditions (constant ones are added inside the tendency
// kernels): after every tendency launch of the stage, while the state buffer still holds the old state and the second buffer
// the new one; one launch per Bounded dimension that carries an array Flux, in the reference's x, y, z order
template <class FT>
static void model_boundary_fluxes(ob200_model* m, const Substep<FT>& ss) {
    const GridD<FT>& g = gridD<FT>(m->grid);
    for (int d = 0; d < 3; ++d) {
        if (g.topo[d] != OB_BOUNDED) continue;
        BoundaryFluxes<FT> a;
        a.n = 0;
        a.ss = ss;
        for (int q = 0; q < m->nf; ++q) {
            const ob200_field* f = m->F[q].get();
            const FT* lo = f->bcs[2 * d].kind == OB200_BC_FLUX ? (const FT*)f->bcv[2 * d] : nullptr;
            const FT* hi = f->bcs[2 * d + 1].kind == OB200_BC_FLUX ? (const FT*)f->bcv[2 * d + 1] : nullptr;
            if (!lo && !hi) continue;
            const int k = a.n++;
            a.comp[k] = std::min(q, 3);
            a.Q[k][0] = lo; a.Q[k][1] = hi;
            a.Gn[k] = m->Gn[q]->template p0<FT>();
            a.Gm[k] = m->Gm[q]->template p0<FT>();
            a.psi[k] = f->template p0<FT>();
            a.psi_new[k] = ss.mode == SUB_NONE ? nullptr : f->template alt0<FT>();
        }
        if (a.n) {
            ScopedPhase ph("boundary_flux");
            launch_boundary_fluxes<FT>(g, d, a);
        }
    }
}

template <class FT>
static void model_tendencies(ob200_model* m, const Substep<FT>& ss) {
    Phys<FT>& P = physOf<FT>(m);
    const FT* U[3] = {m->F[0]->template p0<FT>(), m->F[1]->template p0<FT>(), m->F[2]->template p0<FT>()};
    const FT* pHY = m->pHY ? m->pHY->template p0<FT>() : nullptr;
    const Buoy<FT> b = model_buoyancy<FT>(m);
    // The launches of the prognostic fields are independent (each reads the old state and writes its own G^n and
    // new-state buffer), so they go to side streams forked from the library stream: the tail of one launch (its last,
    // partly filled wave of blocks) overlaps the head of the next instead of leaving SMs idle four times per stage.
    cudaStream_t* side = m->side;
    cudaEvent_t& ev_fork = m->ev_fork;
    cudaEvent_t* ev_join = m->ev_join;
    const bool fork = m->use_fast && m->nf > 1;
    if (fork && !ev_fork) {
        OB_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
        for (int q = 0; q < 3; ++q) {
            OB_CUDA(cudaStreamCreateWithFlags(&side[q], cudaStreamNonBlocking));
            OB_CUDA(cudaEventCreateWithFlags(&ev_join[q], cudaEventDisableTiming));
        }
    }
    ScopedPhase ph("tendency");
    // all fields in one persistent launch (tendency_fused.cu) when the configuration allows; `first` = fields it handled
    int first = 0;
    if (m->use_fast && m->nf >= 3) {
        FusedFields<FT> ff;
        ff.nf = m->nf; ff.pHY = pHY; ff.ss = ss;
        for (int q = 0; q < m->nf && q < FUSED_MAXF; ++q) {
            ob200_field* f = m->F[q].get();
            ff.state[q] = f->template p0<FT>();
            ff.Gm[q] = m->Gm[q]->template p0<FT>();
            ff.Gn[q] = m->Gn[q]->template p0<FT>();
            ff.nw[q] = ss.mode == SUB_NONE ? nullptr : f->template alt0<FT>();
            ff.fbc[q] = constant_flux_bcs<FT>(f);
        }
        // a closure the fused kernel does not evaluate itself (LES closures; any closure on the triply periodic variant): its flux
        // divergence alone goes into G^n through the general shared-face kernel, and the fused kernel adds everything else
        if (fz::supported<FT>(P, m->nf) == 2 && closure_only_supported<FT>(P)) {
            model_halo_join(m);
            const int nfused = 3 + std::min(m->nf - 3, 1);
            const Substep<FT> none{SUB_NONE, FT(0), FT(0), FT(0)};
            for (int q = 0; q < nfused; ++q)
                launch_tendency_general<FT>(P, q, U, ff.state[q], pHY, b, ff.fbc[q], ff.Gn[q], ff.Gm[q], nullptr, none, true);
            ff.accumulate = true;
        }
        // background terms of the fused fields: - div(U_bg, ψ) - div(U, ψ_bg) alone into G^n (onto the closure's part), for the
        // accumulate form to add the rest; it reads the velocities' y halos, so after the exchange has landed.  The variant
        // without a tracer has no accumulate form: that model takes the per-field kernels
        bool bg = false;
        for (int q = 0; q < 3 + std::min(m->nf - 3, 1); ++q) bg = bg || has_background(P, q);
        if (bg && m->nf > 3 && fz::supported<FT>(P, m->nf) && background_only_supported<FT>(P)) {
            model_halo_join(m);
            const Substep<FT> none{SUB_NONE, FT(0), FT(0), FT(0)};
            for (int q = 0; q < 4; ++q)
                launch_tendency_general<FT>(P, q, U, ff.state[q], pHY, b, ff.fbc[q], ff.Gn[q], ff.Gm[q], nullptr, none, false,
                                            ff.accumulate ? 2 : 1);
            ff.gn_terms = true;
        }
        if (bg && !ff.gn_terms) {
            // no fused launch: the per-field kernels below add the background terms themselves
        } else if (m->halo_pending) {
            // the neighbour exchange of the previous stage is still in flight on the halo stream: tile rows that read only rows
            // this rank owns go first, the boundary tile rows once the exchange has landed
            first = fz::launch<FT>(P, ff, 1);
            model_halo_join(m);
            if (first) fz::launch<FT>(P, ff, 2);
            else first = fz::launch<FT>(P, ff, 0);
        } else {
            first = fz::launch<FT>(P, ff, 0);
        }
    }
    model_halo_join(m);
    if (fork) OB_CUDA(cudaEventRecord(ev_fork, g_stream));
    bool lane_forked[3] = {false, false, false};        // a side stream waits for the fork event before its first launch
    for (int q = first; q < m->nf; ++q) {
        ob200_field* f = m->F[q].get();
        const FluxBC<FT> fbc = constant_flux_bcs<FT>(f);
        FT* newp = ss.mode == SUB_NONE ? nullptr : f->template alt0<FT>();
        bool done = false;
        const int lane = fork ? q % 4 : 0;               // lane 0 = the library stream itself
        if (lane > 0) {
            if (!lane_forked[lane - 1]) { OB_CUDA(cudaStreamWaitEvent(side[lane - 1], ev_fork, 0)); lane_forked[lane - 1] = true; }
            g_override = side[lane - 1];
        }
        try {
            if (m->use_fast)
                done = launch_tendency_fast<FT>(P, q, U, f->template p0<FT>(), pHY, m->Gn[q]->template p0<FT>(),
                                                m->Gm[q]->template p0<FT>(), newp, ss);
            if (!done)
                launch_tendency_general<FT>(P, q, U, f->template p0<FT>(), pHY, b, fbc, m->Gn[q]->template p0<FT>(),
                                            m->Gm[q]->template p0<FT>(), newp, ss);
        } catch (...) { g_override = nullptr; throw; }
        g_override = nullptr;
    }
    if (fork)
        for (int q = 0; q < 3 && q + 1 < m->nf; ++q) {
            OB_CUDA(cudaEventRecord(ev_join[q], side[q]));
            OB_CUDA(cudaStreamWaitEvent(g_stream, ev_join[q], 0));
        }
    model_boundary_fluxes<FT>(m, ss);
    if (ss.mode != SUB_NONE) {
        // the out-of-place substep wrote the new state into the second buffer: swap.  Cells the
        // kernels never write (wall faces, outer halos of Bounded dims) are refreshed by the halo
        // fill that always follows, or are never read, exactly as in the reference.
        for (int q = 0; q < m->nf; ++q) std::swap(m->F[q]->base, m->F[q]->alt);
    }
}
// implicit_step! of every prognostic field right after its substep (runge_kutta_3.jl:178-185, quasi_adams_bashforth_2.jl:137-144)
template <class FT>
static void model_implicit_step(ob200_model* m, FT dt) {
    if (!m->desc.closure_vertically_implicit) return;
    ScopedPhase ph("closure");
    const GridD<FT>& g = gridD<FT>(m->grid);
    Phys<FT>& P = physOf<FT>(m);
    for (int q = 0; q < m->nf; ++q)
        launch_implicit_vertical_diffusion<FT>(g, m->F[q]->template p0<FT>(), m->ivd_scratch->template p0<FT>(),
                                               q < 3 ? P.nu : P.kappa[q - 3], dt, q == 2);
}

extern "C" int32_t ob200_model_calculate_tendencies(ob200_model* m) {
    API_BEGIN
    if (m->grid->ftype == OB200_F32) { Substep<float> s{SUB_NONE, 0, 0, 0}; model_tendencies<float>(m, s); }
    else { Substep<double> s{SUB_NONE, 0, 0, 0}; model_tendencies<double>(m, s); }
    API_END
}

template <class FT>
static void model_pressure_step(ob200_model* m, FT dt, bool tracers_too = false, bool fused = false) {
    // calculate_pressure_correction! + pressure_correct_velocities! (pressure_correction.jl:10-56).
    // Inside time_step! the tracers' halos are filled here as well (they do not change until the next
    // substep), which lets the update_state! that follows merge its two halo fills into one.
    // fused: the solver reads the predictor velocities and the correction reads pNHS with periodic wrap-around,
    // so neither fill is needed; the correction kernel stores the halo images of u, v, w and pNHS.
    const GridD<FT>& g = gridD<FT>(m->grid);
    const int dc = fused ? single_comm_dim(g) : -1;      // slab-decomposed dimension of a fused stage, if any
    auto exchange_one = [&](ob200_field* f, bool need_lo, bool need_hi) {
        ScopedPhase ph("halo");
        HaloBatch<FT> hb;
        hb.n = 1;
        halo_entry<FT>(hb, 0, f);
        launch_exchange_planes<FT>(g, hb, dc, 1, need_lo, need_hi);
    };
    if (!fused) { ScopedPhase ph("halo"); model_fill_state_halos<FT>(m, 0, tracers_too ? m->nf : 3); }
    // the divergence needs the velocity normal to the slab boundary one plane beyond it: the neighbour's first plane
    else if (dc >= 0) exchange_one(m->F[dc].get(), false, true);
    { ScopedPhase ph("poisson");
      solve_for_pressure_T<FT>(m->solver.get(), m->pNHS.get(), (double)dt, m->F[0].get(), m->F[1].get(), m->F[2].get()); }
    ob200_field* pn = m->pNHS.get();
    if (!fused) { ScopedPhase ph("halo"); fill_halos<FT>(&pn, 1); }
    // the pressure gradient at the first face of the slab needs the neighbour's last plane of pNHS
    else if (dc >= 0) exchange_one(pn, true, false);
    ScopedPhase ph("pressure_correct");
    launch_pressure_correct<FT>(g, m->F[0]->template p0<FT>(), m->F[1]->template p0<FT>(),
                                m->F[2]->template p0<FT>(), m->pNHS->template p0<FT>(), dt, fused);
}
extern "C" int32_t ob200_model_pressure_project(ob200_model* m, double dt) {
    API_BEGIN
    if (m->grid->ftype == OB200_F32) model_pressure_step<float>(m, (float)dt);
    else model_pressure_step<double>(m, dt);
    API_END
}

template <class FT>
static void model_time_step(ob200_model* m, double dt_in, bool euler) {
    FT dt = (FT)dt_in;
    if (m->desc.timestepper == OB200_TS_RK3) {
        // runge_kutta_3.jl:81-152; γ, ζ stored as FT (:57-66)
        if (m->iteration == 0) model_update_state<FT>(m);
        const FT g1 = FT(8.0 / 15.0), g2 = FT(5.0 / 12.0), g3 = FT(3.0 / 4.0);
        const FT z2 = FT(-17.0 / 60.0), z3 = FT(-5.0 / 12.0);
        FT sdt[3] = {g1 * dt, (g2 + z2) * dt, (g3 + z3) * dt};
        Substep<FT> ss[3] = {{SUB_RK3_FIRST, dt, dt * g1, 0}, {SUB_RK3, dt, g2, z2}, {SUB_RK3, dt, g3, z3}};
        const bool fused = model_fused_periodic<FT>(m);
        for (int s = 0; s < 3; ++s) {
            model_tendencies<FT>(m, ss[s]);
            model_implicit_step<FT>(m, sdt[s]);
            const bool hy = fused && model_hydrostatic_async_begin<FT>(m);
            model_pressure_step<FT>(m, sdt[s], true, fused);
            m->time += (double)sdt[s];
            if (s < 2) for (int q = 0; q < m->nf; ++q) std::swap(m->Gn[q]->base, m->Gm[q]->base);   // store_tendencies!
            if (hy) model_hydrostatic_async_end(m);
            model_update_state_after_projection<FT>(m, fused, hy, s < 2);
        }
        m->iteration += 1;
    } else {
        // quasi_adams_bashforth_2.jl:70-104
        euler = euler || (dt_in != m->previous_dt);
        FT chi = euler ? FT(-0.5) : (FT)m->desc.chi;
        if (euler)
            for (int q = 0; q < m->nf; ++q)
                OB_CUDA(cudaMemsetAsync(m->Gm[q]->base, 0, gtotal(m->grid) * sizeof(FT), stream()));
        m->previous_dt = dt_in;
        if (m->iteration == 0) model_update_state<FT>(m);
        Substep<FT> ss{SUB_AB2, dt, FT(1.5) + chi, FT(0.5) + chi};
        const bool fused = model_fused_periodic<FT>(m);
        model_tendencies<FT>(m, ss);
        model_implicit_step<FT>(m, dt);
        const bool hy = fused && model_hydrostatic_async_begin<FT>(m);
        model_pressure_step<FT>(m, dt, true, fused);
        for (int q = 0; q < m->nf; ++q) std::swap(m->Gn[q]->base, m->Gm[q]->base);
        m->time += (double)dt;
        m->iteration += 1;
        if (hy) model_hydrostatic_async_end(m);
        model_update_state_after_projection<FT>(m, fused, hy);
    }
}
extern "C" int32_t ob200_model_time_step(ob200_model* m, double dt, int32_t euler) {
    API_BEGIN
    if (m->grid->ftype == OB200_F32) model_time_step<float>(m, dt, euler != 0);
    else model_time_step<double>(m, dt, euler != 0);
    API_END
}

extern "C" int32_t ob200_model_clock(const ob200_model* m, double* t, int64_t* it) {
    if (t) *t = m->time;
    if (it) *it = m->iteration;
    return 0;
}
extern "C" int32_t ob200_model_previous_time_step(const ob200_model* m, double* dt) {
    if (!m || !dt) return 1;
    *dt = m->previous_dt;
    return 0;
}
extern "C" int32_t ob200_model_set_clock(ob200_model* m, double t, int64_t it, double pdt) {
    m->time = t; m->iteration = it; m->previous_dt = pdt;
    return 0;
}

extern "C" int32_t ob200_model_diagnostics(ob200_model* m, double* maxdiv, double* ke) {
    API_BEGIN
    double* r = red_buf();
    double h[4];
    if (maxdiv) {
        if (m->grid->ftype == OB200_F32)
            launch_max_divergence<float>(m->grid->g32, m->F[0]->p0<float>(), m->F[1]->p0<float>(), m->F[2]->p0<float>(), r);
        else
            launch_max_divergence<double>(m->grid->g64, m->F[0]->p0<double>(), m->F[1]->p0<double>(), m->F[2]->p0<double>(), r);
        OB_CUDA(cudaMemcpyAsync(h, r, sizeof(h), cudaMemcpyDeviceToHost, stream()));
        OB_CUDA(cudaStreamSynchronize(stream()));
        *maxdiv = h[3] > 0 ? (0.0 / 0.0) : h[2];
    }
    if (ke) {
        double acc = 0;
        for (int q = 0; q < 3; ++q) {
            double s2 = 0;
            if (ob200_field_reduce(m->F[q].get(), nullptr, &s2, nullptr, nullptr)) throw Error(ob::g_err);
            acc += s2;
        }
        *ke = 0.5 * acc;
    }
    API_END
}

// maximum(abs, parent(u)), maximum(abs, parent(v)), maximum(abs, parent(w)): the three device reductions of
// cell_advection_timescale (Utils/cell_advection_timescale.jl:4-21; the reference reduces over the PARENT arrays, halos
// included).  The host divides the grid's minimum spacings by them (TimeStepWizard, Simulations/time_step_wizard.jl:78-95).
extern "C" int32_t ob200_model_max_abs_velocities(ob200_model* m, double out[3]) {
    API_BEGIN
    static double* buf = nullptr;
    if (!buf) OB_CUDA(cudaMalloc(&buf, 12 * sizeof(double)));
    const ob200_grid_desc& D = m->grid->desc;
    for (int q = 0; q < 3; ++q) {
        const ob200_field* f = m->F[q].get();
        int lo[3], n[3];
        for (int d = 0; d < 3; ++d) {
            const bool flat = D.topology[d] == OB200_FLAT;
            lo[d] = flat ? 1 : 1 - D.H[d];
            n[d] = flat ? 1 : D.N[d] + 2 * D.H[d] + ((f->loc[d] == OB200_FACE && D.topology[d] == OB200_BOUNDED) ? 1 : 0);
        }
        if (m->grid->ftype == OB200_F32) launch_reduce_box<float>(m->grid->g32, f->p0<float>(), lo, n, buf + 4 * q);
        else launch_reduce_box<double>(m->grid->g64, f->p0<double>(), lo, n, buf + 4 * q);
    }
    double h[12];
    OB_CUDA(cudaMemcpyAsync(h, buf, sizeof(h), cudaMemcpyDeviceToHost, stream()));
    OB_CUDA(cudaStreamSynchronize(stream()));
    for (int q = 0; q < 3; ++q) out[q] = h[4 * q + 3] > 0 ? (0.0 / 0.0) : h[4 * q + 2];
    API_END
}

// number of cached tensor-map encodings (tests: the cache is bounded, entries die with the buffers they describe)
extern "C" int64_t ob200_debug_cached_tensor_maps(void) { return (int64_t)ob::tmau::cached_maps(); }

// knob used by tests to force the general kernels
extern "C" int32_t ob200_model_use_fast_kernels(ob200_model* m, int32_t on) { m->use_fast = on != 0; return 0; }

// ---- profiling knobs (not part of the reference interface; bench evidence only) ---------------
extern "C" int32_t ob200_profile_enable(int32_t on) {
    ob::g_profile = on != 0;
    return 0;
}
extern "C" int32_t ob200_profile_reset(void) {
    API_BEGIN
    resolve_phases();
    ob::g_phases.clear();
    API_END
}
extern "C" int32_t ob200_profile_query(const char* phase, double* total_ms, int64_t* count) {
    API_BEGIN
    resolve_phases();
    auto it = ob::g_phases.find(phase);
    if (total_ms) *total_ms = it == ob::g_phases.end() ? 0.0 : it->second.total_ms;
    if (count) *count = it == ob::g_phases.end() ? 0 : it->second.count;
    API_END
}

// ---- slab decomposition over several GPUs (reference: src/Distributed/multi_architectures.jl:7-137) -----
namespace ob { namespace comm {
void unique_id(char out[128]); void init(int nranks, int rank, const char id[128]); void destroy();
int rank(); int size(); bool active(); void allreduce_f64(double* buf, size_t n, bool max);
} }
extern "C" int32_t ob200_comm_unique_id(char out[128]) {
    API_BEGIN
    ob::comm::unique_id(out);
    API_END
}
extern "C" int32_t ob200_comm_init(int32_t nranks, int32_t rank, const char id[128]) {
    API_BEGIN
    ensure_device();
    ob::comm::init(nranks, rank, id);
    API_END
}
extern "C" int32_t ob200_comm_destroy(void) {
    API_BEGIN
    ob::comm::destroy();
    API_END
}
// sum (op = 0) or max (op = 1) of n host doubles over all ranks (diagnostics: KE, max |div|, CFL)
extern "C" int32_t ob200_comm_allreduce(double* values, int32_t n, int32_t op) {
    API_BEGIN
    if (!ob::comm::active()) return 0;
    double* r = red_buf();
    if (n > 8) throw Error("at most 8 values");
    OB_CUDA(cudaMemcpyAsync(r, values, n * sizeof(double), cudaMemcpyHostToDevice, stream()));
    ob::comm::allreduce_f64(r, n, op == 1);
    OB_CUDA(cudaMemcpyAsync(values, r, n * sizeof(double), cudaMemcpyDeviceToHost, stream()));
    OB_CUDA(cudaStreamSynchronize(stream()));
    API_END
}
