// ccu_group.cu - multi-GPU entry points of libchunkycu.so (include/chunkycu.h "multi-GPU"): samples-per-pixel split over the
// GPUs of one box, one NCCL reduce-scatter of the window sums over NVLink, per-GPU read-back of its share over its own PCIe
// link and a parallel merge into Chunky's sample buffer (SURVEY.md 8e; OpenClPathTracingRenderer.java:164-173).
//
// NCCL is bound at run time (dlopen "libnccl.so.2"): a single-GPU host never needs it, and a process that already carries an
// NCCL (e.g. a Python host with torch loaded) shares that copy instead of getting a second one.
#include <dlfcn.h>
#include <nccl.h>

#include <cstdio>
#include <cstdlib>
#include <memory>

#include "ccu_host.h"

using ccu_host::DeviceGuard;
using ccu_host::fail;

namespace {

struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*ReduceScatter)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    std::string why;
};

NcclApi *nccl() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        // CCU_NCCL_LIB names the copy to use; a process that will also load another NCCL user (a Python host with torch)
        // must end up with ONE libnccl.so.2 that is new enough for both - the loader shares by soname whichever came first
        // (chunkyclplugin_b200/native.py points CCU_NCCL_LIB at the NCCL bundled with torch when there is one).
        const char *names[] = {getenv("CCU_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char *n : names) {
            if (!n || !*n) continue;
            api.lib = dlopen(n, RTLD_NOW | RTLD_LOCAL);
            if (api.lib) break;
        }
        if (!api.lib) { api.why = std::string("libnccl.so.2 not loadable: ") + dlerror(); return; }
        auto sym = [&](const char *n) { void *p = dlsym(api.lib, n); if (!p && api.why.empty()) api.why = std::string("NCCL symbol missing: ") + n; return p; };
        api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
        api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
        api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
        api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
        api.ReduceScatter = (decltype(api.ReduceScatter))sym("ncclReduceScatter");
        api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
        api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
        api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    });
    return &api;
}

#define NC(call)                                                                                                         \
    do {                                                                                                                 \
        ncclResult_t r_ = (call);                                                                                        \
        if (r_ != ncclSuccess) return fail(CCU_ECUDA, "%s: %s", #call, nccl()->GetErrorString ? nccl()->GetErrorString(r_) : "NCCL error"); \
    } while (0)

struct Member {
    ccu_ctx *ctx = nullptr;
    bool owned = false;
    ncclComm_t comm = nullptr;
    int rank = 0;                      // global rank: which passes (p mod world) and which share of the buffer this GPU owns
    ccu_host::DevBuf<float> share;     // reduce-scatter result: floats [rank * share.n, (rank + 1) * share.n) of the window sum
    ccu_host::Event ev0, ev1;
};

}  // namespace

struct ccu_group {
    int world = 1;
    std::vector<Member> local;
    std::mutex mu;
    int width = 0, height = 0;
    int window_total = 0;               // passes of all ranks in the open window
    int reduced_total = 0;              // passes of the window whose sum sits in the share buffers (reduced, not yet merged)
    bool reduced_equal = true;          // ... and whether that sum is a sum of means (equal pass counts) or of window sums
    float render_ms = 0, reduce_ms = 0;
    // asynchronous share merge (ccu_group_render_merge_async): the reduce-scatter result sits in the share buffers, so the next
    // window may render while the shares travel to the host and are merged
    ccu_host::MergeJob merge;
};

namespace {

int passes_of_rank(int n_total_before, int n_new, int rank, int world) {
    // passes are numbered globally across the window: pass p goes to rank p mod world
    int cnt = 0;
    for (int p = n_total_before; p < n_total_before + n_new; p++) cnt += (p % world == rank);
    return cnt;
}

void free_member(Member &m) {
    if (!m.ctx) return;
    DeviceGuard g(m.ctx->device);
    if (m.comm && nccl()->CommDestroy) nccl()->CommDestroy(m.comm);
    if (m.owned) ccu_ctx_destroy(m.ctx);
    m = Member();
}

int init_member_events(Member &m) {
    DeviceGuard g(m.ctx->device);
    CU(m.ev0.create(cudaEventDefault));
    CU(m.ev1.create(cudaEventDefault));
    return CCU_OK;
}

}  // namespace

extern "C" {

int ccu_group_unique_id(uint8_t id[CCU_UNIQUE_ID_BYTES]) {
    static_assert(sizeof(ncclUniqueId) == CCU_UNIQUE_ID_BYTES, "ncclUniqueId size");
    if (!id) return fail(CCU_EINVAL, "ccu_group_unique_id: null");
    NcclApi *n = nccl();
    if (!n->why.empty()) return fail(CCU_ENODEVICE, "%s", n->why.c_str());
    ncclUniqueId u;
    NC(n->GetUniqueId(&u));
    memcpy(id, &u, sizeof u);
    return CCU_OK;
}

int ccu_group_create(const int32_t *devices, int32_t n, ccu_group **out) {
    if (!out) return fail(CCU_EINVAL, "ccu_group_create: null out");
    *out = nullptr;
    if (!devices || n < 1 || n > 64) return fail(CCU_EINVAL, "ccu_group_create: bad device list (n=%d)", n);
    for (int i = 0; i < n; i++)
        for (int j = 0; j < i; j++)
            if (devices[i] == devices[j]) return fail(CCU_EINVAL, "ccu_group_create: device %d listed twice", devices[i]);
    NcclApi *api = nccl();
    if (n > 1 && !api->why.empty()) return fail(CCU_ENODEVICE, "%s", api->why.c_str());
    std::unique_ptr<ccu_group> g(new ccu_group());
    g->world = n;
    g->local.resize(n);
    int rc = CCU_OK;
    for (int i = 0; i < n && rc == CCU_OK; i++) {
        rc = ccu_ctx_create(devices[i], &g->local[i].ctx);
        g->local[i].owned = true;
        g->local[i].rank = i;
        if (rc == CCU_OK) rc = init_member_events(g->local[i]);
    }
    if (rc == CCU_OK && n > 1) {
        // peer access: scene replication and NCCL's P2P transport over NVLink
        for (int i = 0; i < n; i++) {
            DeviceGuard dg(devices[i]);
            for (int j = 0; j < n; j++) {
                if (i == j) continue;
                int can = 0;
                cudaDeviceCanAccessPeer(&can, devices[i], devices[j]);
                if (can) {
                    cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
                    if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                }
            }
        }
        std::vector<ncclComm_t> comms(n);
        std::vector<int> devs(devices, devices + n);
        ncclResult_t r = api->CommInitAll(comms.data(), n, devs.data());
        if (r != ncclSuccess) rc = fail(CCU_ECUDA, "ncclCommInitAll: %s", api->GetErrorString(r));
        else for (int i = 0; i < n; i++) g->local[i].comm = comms[i];
    }
    if (rc != CCU_OK) {
        std::string keep = ccu_host::last_error();
        for (auto &m : g->local) free_member(m);
        return fail(rc, "%s", keep.c_str());
    }
    *out = g.release();
    return CCU_OK;
}

int ccu_group_join(ccu_ctx *ctx, const uint8_t id[CCU_UNIQUE_ID_BYTES], int32_t rank, int32_t world, ccu_group **out) {
    if (!out) return fail(CCU_EINVAL, "ccu_group_join: null out");
    *out = nullptr;
    if (!ctx || world < 1 || rank < 0 || rank >= world || (world > 1 && !id)) return fail(CCU_EINVAL, "ccu_group_join: bad argument (rank %d of %d)", rank, world);
    NcclApi *api = nccl();
    if (world > 1 && !api->why.empty()) return fail(CCU_ENODEVICE, "%s", api->why.c_str());
    std::unique_ptr<ccu_group> g(new ccu_group());
    g->world = world;
    g->local.resize(1);
    Member &m = g->local[0];
    m.ctx = ctx;
    m.owned = false;
    m.rank = rank;
    int rc = init_member_events(m);
    if (rc == CCU_OK && world > 1) {
        DeviceGuard dg(ctx->device);
        ncclUniqueId u;
        memcpy(&u, id, sizeof u);
        ncclResult_t r = api->CommInitRank(&m.comm, world, u, rank);
        if (r != ncclSuccess) rc = fail(CCU_ECUDA, "ncclCommInitRank: %s", api->GetErrorString(r));
    }
    if (rc != CCU_OK) {
        std::string keep = ccu_host::last_error();
        free_member(m);
        return fail(rc, "%s", keep.c_str());
    }
    *out = g.release();
    return CCU_OK;
}

int ccu_group_destroy(ccu_group *g) {
    if (!g) return CCU_OK;
    ccu_group_render_merge_wait(g);
    for (auto &m : g->local) free_member(m);
    delete g;
    return CCU_OK;
}

int ccu_group_size(ccu_group *g, int32_t *world, int32_t *local_members) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_size: null group");
    if (world) *world = g->world;
    if (local_members) *local_members = (int32_t)g->local.size();
    return CCU_OK;
}

int ccu_group_member(ccu_group *g, int32_t i, ccu_ctx **ctx) {
    if (!g || !ctx || i < 0 || i >= (int)g->local.size()) return fail(CCU_EINVAL, "ccu_group_member: bad argument");
    *ctx = g->local[i].ctx;
    return CCU_OK;
}

int ccu_group_replicate_scene(ccu_group *g) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_replicate_scene: null group");
    std::lock_guard<std::mutex> lk(g->mu);
    for (size_t i = 1; i < g->local.size(); i++) {
        int rc = ccu_host::replicate_scene(g->local[0].ctx, g->local[i].ctx);
        if (rc != CCU_OK) return rc;
    }
    return CCU_OK;
}

int ccu_group_camera_set(ccu_group *g, int32_t projector_type, const float *settings, int64_t n) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_camera_set: null group");
    for (auto &m : g->local) {
        int rc = ccu_camera_set(m.ctx, projector_type, settings, n);
        if (rc != CCU_OK) return rc;
    }
    return CCU_OK;
}

int ccu_group_render_set_params(ccu_group *g, const ccu_render_params *p) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_render_set_params: null group");
    for (auto &m : g->local) {
        int rc = ccu_render_set_params(m.ctx, p);
        if (rc != CCU_OK) return rc;
    }
    return CCU_OK;
}

int ccu_group_render_begin(ccu_group *g, int32_t width, int32_t height) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_render_begin: null group");
    std::lock_guard<std::mutex> lk(g->mu);
    for (auto &m : g->local) {
        {
            std::lock_guard<std::mutex> cl(m.ctx->mu);
            m.ctx->accum_align = (size_t)g->world * 256;      // equal, 1-KiB aligned reduce-scatter shares
        }
        int rc = ccu_render_begin(m.ctx, width, height);
        if (rc != CCU_OK) return rc;
        size_t total;
        {
            std::lock_guard<std::mutex> cl(m.ctx->mu);
            total = m.ctx->accum_floats;
        }
        const size_t share = total / (size_t)g->world;
        if (m.share.n != share) {
            DeviceGuard dg(m.ctx->device);
            CU(m.share.alloc(share));
        }
    }
    g->width = width;
    g->height = height;
    g->window_total = 0;
    g->reduced_total = 0;
    return CCU_OK;
}

int ccu_group_render_passes(ccu_group *g, const int32_t *seeds, int32_t n_passes) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_render_passes: null group");
    if (n_passes < 0 || (n_passes > 0 && !seeds)) return fail(CCU_EINVAL, "ccu_group_render_passes: bad seeds");
    std::lock_guard<std::mutex> lk(g->mu);
    std::vector<int32_t> mine;
    for (auto &m : g->local) {
        mine.clear();
        for (int p = 0; p < n_passes; p++)
            if ((g->window_total + p) % g->world == m.rank) mine.push_back(seeds[p]);
        if (mine.empty()) continue;
        int rc = ccu_render_passes_async(m.ctx, mine.data(), (int32_t)mine.size());   // returns after the enqueue: all GPUs run concurrently
        if (rc != CCU_OK) return rc;
    }
    g->window_total += n_passes;
    return CCU_OK;
}

int ccu_group_render_sync(ccu_group *g) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_render_sync: null group");
    float worst = 0;
    for (auto &m : g->local) {
        int rc = ccu_render_sync(m.ctx);
        if (rc != CCU_OK) return rc;
        float ms = 0;
        rc = ccu_last_kernel_ms(m.ctx, &ms);
        if (rc != CCU_OK) return rc;
        worst = std::max(worst, ms);
    }
    std::lock_guard<std::mutex> lk(g->mu);
    g->render_ms = worst;
    return CCU_OK;
}

// window means -> (sum over GPUs) in the share buffers; closes the window.  Caller holds g->mu.
static int reduce_window_locked(ccu_group *g) {
    const int total = g->window_total;
    if (total == 0) return CCU_OK;
    const int world = g->world;
    const bool equal = total % world == 0;     // every rank rendered total / world passes: the sum of means needs one scale
    NcclApi *api = nccl();
    // 1. window means -> window sums where the ranks' pass counts differ (otherwise folded into the merge weight)
    if (!equal) {
        for (auto &m : g->local) {
            const int mine = passes_of_rank(0, total, m.rank, world);
            std::lock_guard<std::mutex> cl(m.ctx->mu);
            DeviceGuard dg(m.ctx->device);
            ccu_host::scale_window(m.ctx, (float)mine, m.ctx->accum_floats);
            CU(cudaGetLastError());
        }
    }
    // 2. one reduce-scatter over NVLink: rank r receives floats [r * share, (r + 1) * share) of the sum
    if (world > 1) {
        NC(api->GroupStart());
        for (auto &m : g->local) {
            std::lock_guard<std::mutex> cl(m.ctx->mu);
            DeviceGuard dg(m.ctx->device);
            cudaEventRecord(m.ev0, m.ctx->stream);
            ncclResult_t r = api->ReduceScatter(m.ctx->accum[m.ctx->accum_active].p, m.share.p, m.share.n, ncclFloat, ncclSum, m.comm, m.ctx->stream);
            if (r != ncclSuccess) { api->GroupEnd(); return fail(CCU_ECUDA, "ncclReduceScatter: %s", api->GetErrorString(r)); }
        }
        NC(api->GroupEnd());
        for (auto &m : g->local) {
            DeviceGuard dg(m.ctx->device);
            cudaEventRecord(m.ev1, m.ctx->stream);
            m.ctx->launches++;
        }
    } else {
        // one GPU: its window buffer is the result; keep a copy in the share buffer so that the next window may start
        Member &m = g->local[0];
        std::lock_guard<std::mutex> cl(m.ctx->mu);
        DeviceGuard dg(m.ctx->device);
        CU(cudaMemcpyAsync(m.share.p, m.ctx->accum[m.ctx->accum_active].p, m.share.n * sizeof(float), cudaMemcpyDeviceToDevice, m.ctx->stream));
    }
    g->reduced_total = total;
    g->reduced_equal = equal;
    for (auto &m : g->local) ccu_render_reset_window(m.ctx);   // bufferSppReal = 0 (:170)
    g->window_total = 0;
    return CCU_OK;
}

static int finish_reduce_timing(ccu_group *g) {
    float worst = 0;
    for (auto &m : g->local) {
        DeviceGuard dg(m.ctx->device);
        CU(cudaStreamSynchronize(m.ctx->stream));
        float ms = 0;
        if (g->world > 1 && cudaEventElapsedTime(&ms, m.ev0, m.ev1) == cudaSuccess) worst = std::max(worst, ms);
    }
    g->reduce_ms = worst;
    return CCU_OK;
}

int ccu_group_render_reduce(ccu_group *g, int32_t *window_spp) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_render_reduce: null group");
    std::unique_lock<std::mutex> lk(g->mu);
    if (window_spp) *window_spp = g->window_total;
    int rc = g->merge.join(lk);
    if (rc != CCU_OK) return rc;
    rc = reduce_window_locked(g);
    if (rc != CCU_OK) return rc;
    return finish_reduce_timing(g);
}

int ccu_group_render_merge_wait(ccu_group *g) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_render_merge_wait: null group");
    std::unique_lock<std::mutex> lk(g->mu);
    return g->merge.join(lk);
}

// reduce (if the window is still open), then start the read-back of every local share on its GPU's copy stream and hand the merge
// to a worker; returns at once.  Caller holds g->mu through `lk`.
static int group_merge_start(ccu_group *g, std::unique_lock<std::mutex> &lk, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp) {
    int rc = g->merge.join(lk);          // one merge at a time: the share / staging buffers are about to be reused
    if (rc != CCU_OK) return rc;
    if (g->window_total > 0) {
        rc = reduce_window_locked(g);
        if (rc != CCU_OK) return rc;
    }
    const int total = g->reduced_total;
    if (merged_spp) *merged_spp = total;
    if (total == 0) return CCU_OK;
    const int world = g->world;
    const size_t n_img = (size_t)g->width * g->height * 3;
    // every GPU reads its share back over its own PCIe link
    for (auto &m : g->local) {
        ccu_ctx *c = m.ctx;
        DeviceGuard dg(c->device);
        const size_t lo = (size_t)m.rank * m.share.n, hi = std::min(n_img, lo + m.share.n);
        CU(cudaEventRecord(c->window_ev, c->stream));
        CU(cudaStreamWaitEvent(c->copy_stream, c->window_ev, 0));
        if (lo < hi) {
            rc = ccu_host::start_readback(c, m.share.p - lo, lo, hi, c->copy_stream);    // indexed by absolute float offset
            if (rc != CCU_OK) return rc;
        }
    }
    //    sample = (sample * sample_spp + window_mean * total) / (sample_spp + total), window_mean = sum / total (or sum of means / world)
    const double ds = (double)sample_spp, sinv = 1.0 / (double)(sample_spp + total);
    const double dp = g->reduced_equal ? (double)total / (double)world : 1.0;
    g->reduced_total = 0;
    g->merge.start([=] {
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const unsigned merge_threads = std::max(2u, hw / (unsigned)g->local.size());
        std::vector<int> status(g->local.size(), CCU_OK);
        std::vector<std::string> errors(g->local.size());
        auto merge_one = [&](size_t i) {
            Member &m = g->local[i];
            const size_t lo = (size_t)m.rank * m.share.n, hi = std::min(n_img, lo + m.share.n);
            const int st = ccu_host::merge_readback(m.ctx, lo, hi, sample_buffer, ds, dp, sinv, merge_threads);
            if (st != CCU_OK) { status[i] = st; errors[i] = ccu_host::last_error(); }
        };
        if (g->local.size() == 1) {
            merge_one(0);
        } else {
            std::vector<std::thread> th;
            for (size_t i = 0; i < g->local.size(); i++) th.emplace_back(merge_one, i);
            for (auto &t : th) t.join();
        }
        for (size_t i = 0; i < status.size(); i++)
            if (status[i] != CCU_OK) return fail(status[i], "%s", errors[i].c_str());
        return CCU_OK;
    });
    return CCU_OK;
}

int ccu_group_render_merge_async(ccu_group *g, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp) {
    if (!g || !sample_buffer) return fail(CCU_EINVAL, "ccu_group_render_merge_async: null argument");
    if (sample_spp < 0) return fail(CCU_EINVAL, "ccu_group_render_merge_async: negative spp");
    std::unique_lock<std::mutex> lk(g->mu);
    return group_merge_start(g, lk, sample_buffer, sample_spp, merged_spp);
}

int ccu_group_render_merge(ccu_group *g, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp) {
    if (!g || !sample_buffer) return fail(CCU_EINVAL, "ccu_group_render_merge: null argument");
    if (sample_spp < 0) return fail(CCU_EINVAL, "ccu_group_render_merge: negative spp");
    std::unique_lock<std::mutex> lk(g->mu);
    int rc = group_merge_start(g, lk, sample_buffer, sample_spp, merged_spp);
    if (rc != CCU_OK) return rc;
    rc = g->merge.join(lk);
    if (rc != CCU_OK) return rc;
    return finish_reduce_timing(g);
}

int ccu_group_render_end(ccu_group *g) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_render_end: null group");
    int rc = ccu_group_render_merge_wait(g);
    for (auto &m : g->local) {
        const int r = ccu_render_end(m.ctx);
        if (rc == CCU_OK) rc = r;
    }
    std::lock_guard<std::mutex> lk(g->mu);
    g->window_total = 0;
    return rc;
}

int ccu_group_last_ms(ccu_group *g, float *render_ms, float *reduce_ms) {
    if (!g) return fail(CCU_EINVAL, "ccu_group_last_ms: null group");
    std::lock_guard<std::mutex> lk(g->mu);
    if (render_ms) *render_ms = g->render_ms;
    if (reduce_ms) *reduce_ms = g->reduce_ms;
    return CCU_OK;
}

}  // extern "C"
