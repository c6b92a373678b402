// C ABI of libextmcmc_cuda.so (include/extmcmc.h): handle lifetime, device-resident
// workspaces, the block driver that replaces __run! (src/run.jl:64-83) with one CUDA
// graph launch per block of schedule elements, read-back, measurement helpers and the
// NCCL exchange of per-chain partial sums under observation sharding.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/extmcmc.h"
#include "dev_state.cuh"
#include "block_kernels.h"
#include "step_kernels.h"
#include "sweep.h"
#include "user_law.h"

using namespace extmcmc;

namespace {

std::string g_create_error;

// NCCL is resolved at run time so that the library loads (and the single-GPU path
// works) without it, and so that a process that already loaded an NCCL (torch) shares it.
struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t,
                              cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool load(std::string &err) {
        if (lib) return true;
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) { err = std::string("cannot load libnccl: ") + dlerror(); return false; }
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy) {
            err = "libnccl lacks required symbols";
            return false;
        }
        return true;
    }
} g_nccl;

struct Slot {
    StepDesc *h_descs = nullptr;  // pinned
    StepDesc *d_descs = nullptr;
    int cap = 0;
    cudaEvent_t done = nullptr;
    bool in_flight = false;
};

}  // namespace

struct extmcmc_handle {
    extmcmc_config_t cfg{};
    int num_sms = 0;
    size_t l2_bytes = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    DevState d{};
    std::vector<DevUpdate> upd_host;
    std::vector<bool> upd_set;
    bool upd_dirty = true;
    double *obs_dev = nullptr;
    int64_t n_obs_local = 0;
    int64_t n_obs_largest = 0;           // observations of the largest group
    int64_t *goff_dev = nullptr, *glen_dev = nullptr;  // [G] padded group offsets / true lengths
    double *y_dev = nullptr;             // LOGISTIC: responses, padded like the rows of X
    UserLaw ulaw;                        // USER: the compiled law (extmcmc_set_user_law)
    int logi_D = 0;                      // LOGISTIC: padded feature dimension
    unsigned int *tail_counter = nullptr; // CTA counter of the fused sweep tail
    bool tail = false;                   // the obs-mapped sweep finishes the reduction itself
    bool grad_valid = false;             // grad_cur holds d ll/d theta of the CURRENT state
    // Data-sum cache (dev_state.cuh: dsum_cur / dsum_prop).  dcache: the handle keeps one (HIER_NORMAL,
    // observations not sharded, EXTMCMC_DATA_CACHE != 0); dc_valid: dsum_cur holds the per-group data
    // sums of the CURRENT state.
    bool dcache = false, dc_valid = false;
    double *dsum_buf[2] = {nullptr, nullptr};   // the allocations behind d.dsum_cur / d.dsum_prop
    bool any_mala = false;
    bool state_set = false;
    SweepPlan plan{};
    bool plan_valid = false;
    Slot slot[2];
    int next_slot = 0;
    std::map<long long, cudaGraphExec_t> graphs;
    std::map<long long, int64_t> graph_launches;   // kernels per cached graph
    // schedule bookkeeping for the rolling acceptance rate (chain_statistics.jl:53-64)
    int64_t seq_next = 0;
    std::vector<int64_t> ra_iter;   // [NU] mcmciter at which the update last ran (0 = never)
    std::vector<int64_t> acc_tag;   // [NU][W] mcmciter stored in the ring slot (0 = never)
    std::vector<int64_t> haario_M;  // [NU] HaarioTypeAdaptation.M (own-turn counter, adaptation.jl:378)
    // GaussianRandomWalkMix.lambda per update and its schedule f(lambda, N, iter) (adaptation.jl:385,
    // 422-426): evaluated on the host at every readjustment, shipped with the step descriptor
    std::vector<double> lambda;
    std::vector<extmcmc_lambda_fn> lambda_fn;
    std::vector<void *> lambda_user;
    int64_t xseq_next = 0;          // executed steps since handle creation (never reset)
    // persistent block kernels (block_kernels.cu)
    bool blk_planned = false;
    bool res_ok = false, obsblk_ok = false;
    TeamPlan res_plan{};
    ObsBlockPlan obsblk_plan{};
    unsigned long long *blk_go = nullptr;
    unsigned int *blk_counter = nullptr;
    unsigned int *team_sync = nullptr;   // team barrier counters + half-sweep flags (zeroed per launch)
    long long *team_prof = nullptr;      // EXTMCMC_TEAM_PROF: per-CTA cycle breakdown, printed at destroy
    size_t team_sync_cap = 0;
    // replay staging
    double *rp_prop = nullptr, *rp_exp = nullptr;
    size_t rp_prop_cap = 0, rp_exp_cap = 0;
    // instrumentation
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pending, ev_free;
    float sweep_ms = 0.f;
    int64_t sweep_launches = 0;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    std::vector<cudaEvent_t> ev_pool;
    int64_t launches = 0;
    double *flush_buf = nullptr;
    int64_t flush_n = 0;
    double *scratch_ll = nullptr;  // [C]
    double *gsum = nullptr;        // [2][G][C] all-reduced per-group sums of a gradient sweep (obs sharding)
    // asynchronous history fetch
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t fetch_ready = nullptr, fetch_done = nullptr;
    unsigned char *stage = nullptr;   // pinned
    size_t stage_cap = 0;
    int64_t fetch_lo = 0, fetch_hi = 0;
    bool fetch_active = false;
    // fused peer exchange
    void *p2p_region = nullptr;                 // rx[2][W][C] tagged 16-byte cells (exchange.cuh)
    std::vector<void *> p2p_opened;             // peer mappings to close
    // multi-rank
    ncclComm_t comm = nullptr;
    int64_t *n_obs_dev = nullptr;
    bool n_total_known = false;
    std::vector<void *> allocs;
};

namespace {

#define CK(h, call)                                                                      \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);               \
            return e_ == cudaErrorMemoryAllocation ? EXTMCMC_EOOM : EXTMCMC_ECUDA;       \
        }                                                                                \
    } while (0)

#define NK(h, call)                                                                      \
    do {                                                                                 \
        ncclResult_t r_ = (call);                                                        \
        if (r_ != ncclSuccess) {                                                         \
            (h)->err = std::string(#call) + ": " +                                       \
                       (g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "nccl error"); \
            return EXTMCMC_ENCCL;                                                        \
        }                                                                                \
    } while (0)

int32_t fail(extmcmc_t h, int32_t code, const std::string &msg) {
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}

template <typename T>
int32_t dev_alloc(extmcmc_t h, T **out, size_t n) {
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T));
    if (e != cudaSuccess) {
        h->err = std::string("cudaMalloc: ") + cudaGetErrorString(e);
        return EXTMCMC_EOOM;
    }
    h->allocs.push_back(p);
    *out = (T *)p;
    return EXTMCMC_OK;
}

void invalidate_graphs(extmcmc_t h) {
    for (auto &kv : h->graphs) cudaGraphExecDestroy(kv.second);
    h->graphs.clear();
    h->graph_launches.clear();
}

bool obs_sharded(extmcmc_t h) {
    return h->cfg.shard_mode == EXTMCMC_SHARD_OBS && h->cfg.world_size > 1;
}

int32_t ensure_plan(extmcmc_t h) {
    if (h->plan_valid) return EXTMCMC_OK;
    if (h->cfg.law == EXTMCMC_LAW_GSN_IID_1D || h->cfg.law == EXTMCMC_LAW_HIER_NORMAL)
        h->plan = plan_sweep_gsn1d(h->d.C, h->n_obs_largest, h->cfg.sweep_variant, h->num_sms, h->d.G);
    else if (h->cfg.law == EXTMCMC_LAW_GSN_MV)
        h->plan = plan_sweep_gsnmv(h->cfg.obs_dim, h->d.C, h->n_obs_local, h->cfg.sweep_variant, h->num_sms);
    else if (h->cfg.law == EXTMCMC_LAW_LOGISTIC)
        h->plan = plan_sweep_logistic(h->cfg.obs_dim, h->d.C, h->n_obs_local, h->num_sms);
    else if (h->cfg.law == EXTMCMC_LAW_USER) {
        if (!h->ulaw.loaded) return fail(h, EXTMCMC_EINVAL, "no user law: call extmcmc_set_user_law first");
        h->plan = plan_sweep_user(h->ulaw, h->d.C, h->n_obs_local, h->cfg.sweep_variant, h->num_sms);
    } else
        return fail(h, EXTMCMC_EUNSUPPORTED, "law not implemented on the GPU path");
    h->d.S = h->plan.S;
    // fused tail of the obs-mapped 1-D sweep (few chains, many segments): see sweep.h
    h->tail = h->cfg.law == EXTMCMC_LAW_GSN_IID_1D && h->plan.variant == SWEEP_VARIANT_OBS;
    if (const char *e = getenv("EXTMCMC_TAIL")) h->tail = h->tail && atoi(e) != 0;   // diagnostics
    if (h->tail && !h->tail_counter) {
        int32_t rct = dev_alloc(h, &h->tail_counter, 1);
        if (rct) return rct;
        CK(h, cudaMemset(h->tail_counter, 0, sizeof(unsigned int)));
    }
    h->d.use_ssum = (obs_sharded(h) || law_self_finished(h->cfg.law) || h->tail) ? 1 : 0;
    // Gaussian laws: two quantities (second- and first-order sums) x G groups x S segments;
    // logistic and user laws: ll_part[S][C] followed by g_part[S][p][C]
    size_t part_rows = law_self_finished(h->cfg.law) ? (size_t)h->plan.S * (h->cfg.n_params + 1)
                                                     : (size_t)2 * h->d.G * h->plan.S;
    part_rows = std::max(part_rows, (size_t)h->num_sms * 3);   // segments of the observation-mapped block kernel
    part_rows = std::max(part_rows, (size_t)2 * h->d.G * 4);   // members of a team of the team-resident block kernel
    int32_t rc = dev_alloc(h, &h->d.partial, part_rows * h->d.C);
    if (rc) return rc;
    if (obs_sharded(h) && !h->gsum &&
        (h->cfg.law == EXTMCMC_LAW_GSN_IID_1D || h->cfg.law == EXTMCMC_LAW_HIER_NORMAL))
        if ((rc = dev_alloc(h, &h->gsum, (size_t)2 * h->d.G * h->d.C))) return rc;
    {
        const char *e = getenv("EXTMCMC_DATA_CACHE");   // read per plan, so that one process can compare both
        const bool on = !e || atoi(e) != 0;
        h->dcache = on && h->cfg.law == EXTMCMC_LAW_HIER_NORMAL && !obs_sharded(h) && h->d.G <= kDataCacheMaxG;
        if (h->dcache && !h->dsum_buf[0])
            if ((rc = dev_alloc(h, &h->dsum_buf[0], (size_t)2 * h->d.G * h->d.C)) ||
                (rc = dev_alloc(h, &h->dsum_buf[1], (size_t)2 * h->d.G * h->d.C)))
                return rc;
        h->d.dsum_cur = h->dcache ? h->dsum_buf[0] : nullptr;
        h->d.dsum_prop = h->dcache ? h->dsum_buf[1] : nullptr;
        h->dc_valid = false;
    }
    h->plan_valid = true;
    h->blk_planned = false;
    invalidate_graphs(h);
    return EXTMCMC_OK;
}

// ---- data-sum cache: which elements need no sweep ------------------------------------------------
// The data term of HIER_NORMAL depends on theta_1..G only.  An element whose update moves none of
// them (mu, tau) proposes a state with the data sums of the current one; a MALA element that follows
// such elements finds the sums of its current state still in the cache.  kinds[] carries the fact as
// kDataFree on top of the transition kernel id; step_advance is the one place that says what an
// element does to (grad_valid, dc_valid) and is used by the descriptor loop, the graph key, the
// kernel sequence and the end-of-block state alike.
constexpr int kDataFree = 0x100;
int step_kind(extmcmc_t h, int u) {
    const DevUpdate &t = h->upd_host[u];
    int kind = t.kernel;
    if (h->dcache && kind != EXTMCMC_KERNEL_MALA && t.n_coords <= kMaxCoords) {
        bool moves_data = false;
        for (int i = 0; i < t.n_coords; ++i) moves_data = moves_data || t.coords[i] < h->d.G;
        if (!moves_data) kind |= kDataFree;
    }
    return kind;
}
inline bool kind_is_mala(int kind) { return (kind & 0xff) == EXTMCMC_KERNEL_MALA; }
// MALA: returns how the gradient of the current state is obtained (0 = still valid, 1 = sweep,
// 2 = from the cache).  Random walk: 0 = the element sweeps its proposal; 1 = it runs from the cache;
// 2 = the cache is refilled first (gradient sweep of the CURRENT state + per-group reduction -- the
// kernels and the association that fill it on the MALA path, so a data-free element sees the same
// bits whether the sums were kept or recomputed: start of a run, after a checkpoint load, after an
// element that moved a theta_g), then as 1.
int step_advance(bool dcache, int kind, bool &gv, bool &dc) {
    if (kind_is_mala(kind)) {
        const int mode = gv ? 0 : (dc ? 2 : 1);
        if (mode == 1 && dcache) dc = true;   // mala_propose stores the sums it finishes
        gv = true;                            // (an accepted proposal hands its sums over: mala_decide_commit)
        return mode;
    }
    gv = false;
    if (kind & kDataFree) {
        const int mode = dc ? 1 : 2;
        dc = true;
        return mode;
    }
    dc = false;
    return 0;
}

// Which schedule blocks run as ONE persistent kernel (block_kernels.cu) instead of a kernel sequence
// per element.  cfg.sweep_variant: 0 = automatic, 3 = chain-resident kernel whenever it is
// applicable (tests: also with few chains), 4 = observation-mapped block kernel likewise, any
// other value pins the per-step path.
int32_t plan_block_kernels(extmcmc_t h) {
    if (h->blk_planned) return EXTMCMC_OK;
    h->blk_planned = true;
    h->res_ok = h->obsblk_ok = false;
    const int sv = h->cfg.sweep_variant;
    if (sv != 0 && sv != 3 && sv != 4) return EXTMCMC_OK;
    if (const char *e = getenv("EXTMCMC_BLOCK_KERNELS")) if (atoi(e) == 0) return EXTMCMC_OK;   // diagnostics
    const bool gsn1d = h->cfg.law == EXTMCMC_LAW_GSN_IID_1D || h->cfg.law == EXTMCMC_LAW_HIER_NORMAL;
    if (!gsn1d || h->d.n_haario > 0) return EXTMCMC_OK;
    bool all_unif = true, all_unif_or_mala = true;
    for (int u = 0; u < h->cfg.n_updates; ++u) {
        const int kk = h->upd_host[u].kernel;
        if (kk != EXTMCMC_KERNEL_RW_UNIFORM) all_unif = false;
        if (kk != EXTMCMC_KERNEL_RW_UNIFORM && kk != EXTMCMC_KERNEL_MALA) all_unif_or_mala = false;
    }
    // The team-resident kernel is opt-in (sweep_variant 3): measured on B200 it does not beat the
    // per-step kernels -- with observations of the cfg 2 size every CTA-level stream of them is bound
    // by L2 -> SM delivery, and with small data (cfg 4) the FP64-latency-bound scalar phases are not
    // hidden well enough (DESIGN.md, "Persistent block kernels").
    if (all_unif_or_mala && !obs_sharded(h) && sv == 3) {
        h->res_ok = plan_team(h->d, h->upd_host.data(), h->num_sms, true, &h->res_plan);
        if (h->res_ok && getenv("EXTMCMC_TEAM_PROF") && !h->team_prof) {
            int32_t rc = dev_alloc(h, &h->team_prof, (size_t)h->res_plan.n_cta * 8);
            if (rc) return rc;
            CK(h, cudaMemset(h->team_prof, 0, sizeof(long long) * h->res_plan.n_cta * 8));
        }
        if (h->res_ok) {
            const size_t words = team_sync_words(h->res_plan);
            if (words > h->team_sync_cap) {
                int32_t rc = dev_alloc(h, &h->team_sync, words);
                if (rc) return rc;
                h->team_sync_cap = words;
            }
        }
    }
    // The observation-mapped block kernel is opt-in too (sweep_variant 4): with 125 M observations per
    // GPU it gains 2 % over the per-step kernels with the fused exchange, with 500 M per GPU it loses
    // 6 % (two CTAs of 128 registers per SM stream HBM less well than three of 80).
    const bool obs_auto = false;
    if (!h->res_ok && all_unif && h->cfg.law == EXTMCMC_LAW_GSN_IID_1D && h->d.C <= 32 && (sv == 4 || obs_auto) &&
        (!obs_sharded(h) || h->d.p2p)) {
        cudaError_t e = plan_obs_block(h->d, h->upd_host.data(), h->num_sms, h->n_obs_local, &h->obsblk_plan);
        if (e == cudaSuccess) {
            if (!h->blk_go) {
                int32_t rc;
                if ((rc = dev_alloc(h, &h->blk_go, 1)) || (rc = dev_alloc(h, &h->blk_counter, 1))) return rc;
                CK(h, cudaMemset(h->blk_go, 0, sizeof(unsigned long long)));
                CK(h, cudaMemset(h->blk_counter, 0, sizeof(unsigned int)));
            }
            h->obsblk_ok = true;
        } else {
            cudaGetLastError();
        }
    }
    return EXTMCMC_OK;
}

int32_t upload_updates(extmcmc_t h) {
    if (!h->upd_dirty) return EXTMCMC_OK;
    CK(h, cudaMemcpyAsync(h->d.upd, h->upd_host.data(), sizeof(DevUpdate) * h->upd_host.size(),
                          cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    h->upd_dirty = false;
    return EXTMCMC_OK;
}

int32_t ensure_total_obs(extmcmc_t h) {
    if (h->n_total_known) return EXTMCMC_OK;
    if (h->cfg.shard_mode == EXTMCMC_SHARD_OBS && h->cfg.world_size > 1) {
        if (!h->comm) return fail(h, EXTMCMC_EINVAL, "EXTMCMC_SHARD_OBS needs extmcmc_comm_init first");
        int64_t n = h->n_obs_local;
        CK(h, cudaMemcpyAsync(h->n_obs_dev, &n, sizeof n, cudaMemcpyHostToDevice, h->stream));
        NK(h, g_nccl.AllReduce(h->n_obs_dev, h->n_obs_dev, 1, ncclInt64, ncclSum, h->comm, h->stream));
        CK(h, cudaMemcpyAsync(&n, h->n_obs_dev, sizeof n, cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        h->d.n_obs_total = n;
    } else {
        h->d.n_obs_total = h->n_obs_local;
    }
    h->n_total_known = true;
    invalidate_graphs(h);
    return EXTMCMC_OK;
}

// One likelihood sweep (+ cross-rank reduction when the observations are sharded).  Gaussian
// laws read the law constants the proposal kernel left in lawc and leave per-segment sums in
// `partial` (grad: also the first-order sums).  The logistic law reads the parameters from
// `src` ([p][C]) and finishes ll (-> ll_dst) and the gradient (-> grad_dst, may be NULL) itself.
int32_t enqueue_sweep(extmcmc_t h, bool instrument, bool grad = false, const double *src = nullptr,
                      double *ll_dst = nullptr, double *grad_dst = nullptr,
                      const StepDesc *d_descs = nullptr, int k = 0) {
    std::pair<cudaEvent_t, cudaEvent_t> ev{nullptr, nullptr};
    bool tail_done = false;   // the sweep kernel itself reduced (and, with p2p, delivered) the sums
    if (instrument) {
        if (!h->ev_free.empty()) { ev = h->ev_free.back(); h->ev_free.pop_back(); }
        else { CK(h, cudaEventCreate(&ev.first)); CK(h, cudaEventCreate(&ev.second)); }
        CK(h, cudaEventRecord(ev.first, h->stream));
    }
    if (h->cfg.law == EXTMCMC_LAW_GSN_IID_1D || h->cfg.law == EXTMCMC_LAW_HIER_NORMAL) {
        Gsn1dArgs a{};
        a.obs = h->obs_dev; a.goff = h->goff_dev; a.glen = h->glen_dev; a.G = h->d.G;
        // per-chain means: the law constants for the iid law; theta_1..G of the evaluated state
        // itself (src, [p][C]) for the hierarchical law
        a.mu = h->cfg.law == EXTMCMC_LAW_HIER_NORMAL ? src : h->d.lawc;
        if (!a.mu) return fail(h, EXTMCMC_EINVAL, "internal: sweep without a source state");
        a.C = h->d.C; a.partial = h->d.partial; a.S = h->plan.S;
        tail_done = h->tail && !grad;
        if (tail_done) {
            const bool push = obs_sharded(h) && h->d.p2p && d_descs;
            a.tail_mode = push ? 2 : 1;
            a.tail_counter = h->tail_counter; a.ssum = h->d.ssum;
            a.peer_rx = h->d.peer_rx;
            a.rank = h->cfg.rank; a.world = h->cfg.world_size;
            a.descs = d_descs; a.k = k;
        }
        // a stream that cannot stay in L2 anyway must not evict the chain state (EXTMCMC_L2_HINT=0: off)
        static const bool hint_on = [] { const char *e = getenv("EXTMCMC_L2_HINT"); return !e || atoi(e) != 0; }();
        a.stream_hint = hint_on && (size_t)h->n_obs_local * sizeof(double) > h->l2_bytes / 2 ? 1 : 0;
        launch_sweep_gsn1d(h->plan, a, grad, h->stream);
    } else if (h->cfg.law == EXTMCMC_LAW_LOGISTIC) {
        LogisticArgs a{h->obs_dev, h->y_dev, h->n_obs_local, src, h->cfg.obs_dim, h->d.C, h->d.partial,
                       h->d.partial + (size_t)h->plan.S * h->d.C, h->plan.S, h->plan.n_cta};
        launch_sweep_logistic(h->plan, a, ll_dst, grad_dst, h->stream);
        if (obs_sharded(h)) {
            // every rank holds a slice of the rows of X: sum the per-chain log-likelihoods and the
            // [d][C] gradients over the ranks (SURVEY 2.2, K4: "allreduce of [C] ll and [C x d] grads")
            NK(h, g_nccl.AllReduce(ll_dst, ll_dst, (size_t)h->d.C, ncclFloat64, ncclSum, h->comm, h->stream));
            if (grad_dst)
                NK(h, g_nccl.AllReduce(grad_dst, grad_dst, (size_t)h->cfg.obs_dim * h->d.C, ncclFloat64, ncclSum,
                                       h->comm, h->stream));
        }
        h->launches += h->plan.launches;
        if (instrument) {
            CK(h, cudaEventRecord(ev.second, h->stream));
            h->ev_pending.push_back(ev);
        }
        return EXTMCMC_OK;
    } else if (h->cfg.law == EXTMCMC_LAW_USER) {
        // same contract as the logistic law: the sweep reads the parameters from src and finishes
        // ll (-> ll_dst) and, with grad, the gradient (-> grad_dst) itself; never sharded by observation
        UserSweepArgs a{};
        a.obs = h->obs_dev; a.n_obs = h->n_obs_local; a.theta = src; a.C = h->d.C;
        a.ll_part = h->d.partial; a.g_part = h->d.partial + (size_t)h->plan.S * h->d.C;
        a.err_flag = h->d.err_flag; a.S = h->plan.S;
        CK(h, launch_sweep_user(h->plan, h->ulaw, a, grad, ll_dst, grad_dst, h->stream));
        h->launches += user_sweep_launches(h->ulaw, grad);
        if (instrument) {
            CK(h, cudaEventRecord(ev.second, h->stream));
            h->ev_pending.push_back(ev);
        }
        return EXTMCMC_OK;
    } else {
        launch_sweep_gsnmv(h->plan, h->obs_dev, h->n_obs_local, h->d.lawc, h->d.C, h->d.partial, h->stream);
    }
    h->launches += h->plan.launches;
    if (instrument) {
        CK(h, cudaEventRecord(ev.second, h->stream));
        h->ev_pending.push_back(ev);
    }
    if (obs_sharded(h) && grad) {
        // gradient sweep of a Gaussian law: the consumers (MALA kernels, extmcmc_eval_grad) need the
        // sums per observation group and of both orders, over all ranks
        launch_reduce_group_sums(h->d, h->gsum, h->stream);
        h->launches += 1;
        NK(h, g_nccl.AllReduce(h->gsum, h->gsum, (size_t)2 * h->d.G * h->d.C, ncclFloat64, ncclSum, h->comm,
                               h->stream));
    } else if (obs_sharded(h)) {
        if (h->d.p2p && d_descs) {
            // our own exchange: peer stores + flags (in the sweep's fused tail, or here), wait +
            // ordered sum inside accept_kernel
            if (!tail_done) { launch_reduce_push(h->d, d_descs, k, h->stream); h->launches += 1; }
        } else {
            if (!tail_done) { launch_reduce_partials(h->d, h->stream); h->launches += 1; }
            NK(h, g_nccl.AllReduce(h->d.ssum, h->d.ssum, (size_t)h->d.C, ncclFloat64, ncclSum, h->comm,
                                   h->stream));
        }
    }
    return EXTMCMC_OK;
}

// Kernel sequence of one block.  kinds[k] = transition kernel of schedule element k (host copy
// of the descriptors).  Random-walk element: [propose] sweep accept(+ next RW proposal fused).
// MALA element: [current-state gradient sweep if grad_cur is stale] propose, gradient sweep,
// finalize, accept.  grad_valid is threaded through so that a captured graph and the eager
// path make identical decisions.
// What the gradient consumers see: under observation sharding the all-reduced per-group sums stand
// in for the partial buffer (one "segment" per group).
DevState grad_view(extmcmc_t h) {
    DevState v = h->d;
    if (obs_sharded(h) && !law_self_finished(h->cfg.law)) { v.partial = h->gsum; v.S = 1; }
    return v;
}

int32_t enqueue_steps(extmcmc_t h, const StepDesc *d_descs, const int *kinds, int n_steps,
                      bool instrument, bool &grad_valid, bool &dc_valid) {
    bool fused = false;      // the proposal of element k was already issued by accept(k-1)
    bool cur_prepared = false;  // accept(k-1) already wrote the law constants of the current state
    for (int k = 0; k < n_steps; ++k) {
        int32_t rc;
        // deferred bookkeeping between consecutive elements of this block (step_kernels.cu, run_deferred)
        const int dflags = step_deferral_flags(h->d, k, n_steps);
        const bool next_mala = k + 1 < n_steps && kind_is_mala(kinds[k + 1]);
        const bool next_rw = k + 1 < n_steps && !kind_is_mala(kinds[k + 1]);
        const int mode = step_advance(h->dcache, kinds[k], grad_valid, dc_valid);
        if (kind_is_mala(kinds[k])) {
            const bool logi = law_self_finished(h->cfg.law);   // the sweep finishes ll and gradient
            int finalize_cur = 0;
            DevState gv = grad_view(h);
            if (mode == 1) {
                if (logi) {
                    if ((rc = enqueue_sweep(h, instrument, true, h->d.theta, h->scratch_ll, h->d.grad_cur))) return rc;
                } else {
                    // current-state gradient sweep; its sums are finished inside mala_propose
                    const bool hier = h->cfg.law == EXTMCMC_LAW_HIER_NORMAL;   // no law constants to prepare
                    if (!cur_prepared && !hier) { launch_prepare_current(h->d, h->stream); h->launches += 1; }
                    if ((rc = enqueue_sweep(h, instrument, true, h->d.theta))) return rc;
                    finalize_cur = 1;
                }
            } else if (mode == 2) {
                // the sums of the current state are in the cache: mala_propose finishes them from there
                gv.partial = h->d.dsum_cur; gv.S = 1;
                finalize_cur = 2;
            }
            launch_mala_propose(gv, d_descs, k, finalize_cur, h->scratch_ll, dflags, h->stream);
            gv = grad_view(h);
            if (logi) {
                if ((rc = enqueue_sweep(h, instrument, true, h->d.prop_full, h->d.ll_prop, h->d.grad_prop))) return rc;
            } else {
                if ((rc = enqueue_sweep(h, instrument, true, h->d.prop_full))) return rc;   // finished inside mala_accept
            }
            fused = next_rw;   // the next random-walk proposal rides on this accept kernel
            launch_mala_accept(gv, d_descs, k, logi ? 0 : 1, fused ? 1 : 0, dflags, h->stream);
            h->launches += 2;
            cur_prepared = false;
        } else {
            if (!fused) { launch_propose(h->d, d_descs, k, h->stream); h->launches += 1; }
            const bool from_cache = mode != 0;
            if (mode == 2) {
                if ((rc = enqueue_sweep(h, instrument, true, h->d.theta))) return rc;
                launch_reduce_group_sums(h->d, h->d.dsum_cur, h->stream);
                h->launches += 1;
            }
            if (!from_cache)
                if ((rc = enqueue_sweep(h, instrument, false, h->d.prop_full, h->d.ssum, nullptr, d_descs, k))) return rc;
            fused = next_rw;
            // a MALA element follows and will need the law constants of the (then) current state for
            // its gradient sweep: let this accept kernel write them (fuse_next = 2)
            cur_prepared = next_mala && !law_self_finished(h->cfg.law) && h->cfg.law != EXTMCMC_LAW_HIER_NORMAL;
            launch_accept(h->d, d_descs, k, fused ? 1 : (cur_prepared ? 2 : 0), dflags, h->stream, from_cache);
            h->launches += 1;
        }
    }
    CK(h, cudaGetLastError());
    return EXTMCMC_OK;
}

int32_t collect_events(extmcmc_t h) {
    for (auto &ev : h->ev_pending) {
        float ms = 0.f;
        CK(h, cudaEventElapsedTime(&ms, ev.first, ev.second));
        h->sweep_ms += ms;
        h->sweep_launches += 1;
        h->ev_free.push_back(ev);
    }
    h->ev_pending.clear();
    return EXTMCMC_OK;
}

int32_t run_block_impl(extmcmc_t h, const extmcmc_step_t *steps, int32_t n_steps, int rng_mode,
                       int32_t p_u_max, const double *proposals, const double *exp_draws) {
    if (!h) return EXTMCMC_EINVAL;
    if (n_steps < 0 || (n_steps > 0 && !steps)) return fail(h, EXTMCMC_EINVAL, "bad steps");
    if (n_steps == 0) return EXTMCMC_OK;
    if (!h->obs_dev) return fail(h, EXTMCMC_EINVAL, "no observations uploaded");
    if (!h->state_set) return fail(h, EXTMCMC_EINVAL, "extmcmc_set_state not called");
    for (int u = 0; u < h->cfg.n_updates; ++u)
        if (!h->upd_set[u]) return fail(h, EXTMCMC_EINVAL, "update " + std::to_string(u) + " not set");
    if (n_steps > h->cfg.history_window)
        return fail(h, EXTMCMC_EINVAL, "block longer than history_window");
    if (obs_sharded(h) && !h->comm) return fail(h, EXTMCMC_EINVAL, "EXTMCMC_SHARD_OBS needs extmcmc_comm_init first");
    if (h->cfg.law == EXTMCMC_LAW_USER && h->any_mala && h->ulaw.loaded && !h->ulaw.grad)
        return fail(h, EXTMCMC_EUNSUPPORTED, "MALA needs a user law with a gradient (extmcmc_set_user_law with_grad = 1 or 2)");
    for (int s = 0; s < n_steps; ++s)
        if (steps[s].pidx < 0 || steps[s].pidx >= h->cfg.n_updates || steps[s].mcmciter < 1)
            return fail(h, EXTMCMC_EINVAL, "step out of range");
    CK(h, cudaSetDevice(h->cfg.device));
    int32_t rc;
    if ((rc = ensure_plan(h))) return rc;
    if ((rc = upload_updates(h))) return rc;
    if ((rc = ensure_total_obs(h))) return rc;
    if ((rc = plan_block_kernels(h))) return rc;
    if ((h->res_ok || h->obsblk_ok) && h->dcache) {   // the persistent block kernels sweep for every element
        h->dcache = h->dc_valid = false;
        h->d.dsum_cur = h->d.dsum_prop = nullptr;
    }
    // a history fetch still in flight reads ring slots this block is about to overwrite: order the
    // block after the copy (callers that keep 2 x block_len rows never get here)
    if (h->fetch_active && h->seq_next + n_steps - h->d.H > h->fetch_lo)
        CK(h, cudaStreamWaitEvent(h->stream, h->fetch_done, 0));

    if (h->d.rng_mode != rng_mode) { h->d.rng_mode = rng_mode; invalidate_graphs(h); }
    if (rng_mode == EXTMCMC_RNG_REPLAY) {
        if (!proposals || !exp_draws || p_u_max < 1) return fail(h, EXTMCMC_EINVAL, "replay buffers missing");
        for (int s = 0; s < n_steps; ++s)
            if (h->upd_host[steps[s].pidx].n_coords > p_u_max)
                return fail(h, EXTMCMC_EINVAL, "p_u_max smaller than an update's n_coords");
        const size_t np = (size_t)n_steps * p_u_max * h->d.C, ne = (size_t)n_steps * h->d.C;
        CK(h, cudaStreamSynchronize(h->stream));
        if (np > h->rp_prop_cap) {
            if (h->rp_prop) cudaFree(h->rp_prop);
            CK(h, cudaMalloc(&h->rp_prop, np * sizeof(double)));
            h->rp_prop_cap = np;
        }
        if (ne > h->rp_exp_cap) {
            if (h->rp_exp) cudaFree(h->rp_exp);
            CK(h, cudaMalloc(&h->rp_exp, ne * sizeof(double)));
            h->rp_exp_cap = ne;
        }
        CK(h, cudaMemcpy(h->rp_prop, proposals, np * sizeof(double), cudaMemcpyHostToDevice));
        CK(h, cudaMemcpy(h->rp_exp, exp_draws, ne * sizeof(double), cudaMemcpyHostToDevice));
        h->d.rp_prop = h->rp_prop;
        h->d.rp_exp = h->rp_exp;
        h->d.p_u_max = p_u_max;
    }

    // descriptor slot (double-buffered so the host can prepare block k+1 while k runs)
    const int si = h->next_slot;
    Slot &sl = h->slot[si];
    h->next_slot ^= 1;
    if (sl.in_flight) { CK(h, cudaEventSynchronize(sl.done)); sl.in_flight = false; }
    if (sl.cap < n_steps) {
        if (sl.h_descs) cudaFreeHost(sl.h_descs);
        if (sl.d_descs) cudaFree(sl.d_descs);
        for (auto it = h->graphs.begin(); it != h->graphs.end();) {
            if ((it->first & 1) == si) { cudaGraphExecDestroy(it->second); it = h->graphs.erase(it); }
            else ++it;
        }
        const int cap = std::max(n_steps, 64);
        CK(h, cudaMallocHost(&sl.h_descs, sizeof(StepDesc) * cap));
        CK(h, cudaMalloc(&sl.d_descs, sizeof(StepDesc) * cap));
        sl.cap = cap;
    }
    const int W = h->d.W;
    int n_sweeps = 0;
    {
        bool gv = h->grad_valid, dc = h->dc_valid;
        for (int s = 0; s < n_steps; ++s) {
            StepDesc &sd = sl.h_descs[s];
            const int u = steps[s].pidx;
            const int64_t it = steps[s].mcmciter;
            sd.mcmciter = it;
            sd.seq = h->seq_next + s;
            sd.stat_n = sd.seq + 1;  // GenericChainStats.N starts at 1 (chain_statistics.jl:34)
            sd.xseq = h->xseq_next + s;
            sd.pidx = u;
            sd.first = steps[s].prev_pidx < 0 ? 1 : 0;
            const int64_t prev_it = it - 1 > 1 ? it - 1 : 1;
            sd.ra_prev_valid = (h->ra_iter[u] == prev_it && prev_it != it) ? 1 : 0;
            int64_t &tag = h->acc_tag[(size_t)u * W + (size_t)(it % W)];
            sd.acc_out_valid = (it > W && tag == it - W) ? 1 : 0;
            sd.replay_row = s;
            sd.haario_ready = 0;
            sd.lambda = h->lambda[u];
            sd.pad_ = 0;
            if (h->upd_host[u].adapt_kind == EXTMCMC_ADAPT_HAARIO) {
                // register_only_on_my_turn(::Val{true}, ::Haario): M += 1; time_to_update: M >= k -> M = 0
                if (++h->haario_M[u] >= h->upd_host[u].adapt_every_k) {
                    sd.haario_ready = 1;
                    h->haario_M[u] = 0;
                    // readjust!: rw.lambda = f(rw.lambda, adpt.N, mcmc_iter) with adpt.N already
                    // incremented by this step's registration (adaptation.jl:413,425)
                    if (h->lambda_fn[u]) h->lambda[u] = h->lambda_fn[u](h->lambda[u], sd.stat_n + 1, it, h->lambda_user[u]);
                }
            }
            const bool mala = h->upd_host[u].kernel == EXTMCMC_KERNEL_MALA;
            sd.need_cur_grad = (mala && !gv) ? 1 : 0;
            const int mode = step_advance(h->dcache, step_kind(h, u), gv, dc);
            n_sweeps += mala ? 1 + (mode == 1 ? 1 : 0) : (mode == 1 ? 0 : 1);
            h->ra_iter[u] = it;
            tag = it;
        }
    }

    std::vector<int> kinds(n_steps);
    unsigned long long hash = 1469598103934665603ull;  // FNV-1a over the kernel-kind sequence
    for (int s = 0; s < n_steps; ++s) {
        kinds[s] = step_kind(h, steps[s].pidx);
        hash = (hash ^ (unsigned long long)kinds[s]) * 1099511628211ull;
    }
    hash = (hash ^ (unsigned long long)((h->grad_valid ? 7 : 3) + (h->dc_valid ? 16 : 0))) * 1099511628211ull;
    hash = (hash ^ (unsigned long long)n_steps) * 1099511628211ull;
    const bool instrument = h->cfg.instrument != 0;
    const bool use_graph = h->cfg.use_graphs && !instrument && rng_mode == EXTMCMC_RNG_PHILOX;
    if (h->res_ok || h->obsblk_ok) {
        // the whole block in one persistent kernel
        CK(h, cudaMemcpyAsync(sl.d_descs, sl.h_descs, sizeof(StepDesc) * n_steps, cudaMemcpyHostToDevice, h->stream));
        std::pair<cudaEvent_t, cudaEvent_t> ev{nullptr, nullptr};
        if (instrument) {
            if (!h->ev_free.empty()) { ev = h->ev_free.back(); h->ev_free.pop_back(); }
            else { CK(h, cudaEventCreate(&ev.first)); CK(h, cudaEventCreate(&ev.second)); }
        }
        if (h->res_ok) {
            TeamArgs a{};
            a.d = h->d;
            a.d.dsum_cur = a.d.dsum_prop = nullptr;
            a.d.S = h->res_plan.ts;        // the members of a team are the "segments" of the partial sums
            a.descs = sl.d_descs; a.n_steps = n_steps; a.n_sweeps = n_sweeps;
            a.obs = h->obs_dev; a.goff = h->goff_dev; a.glen = h->glen_dev; a.G = h->d.G;
            a.ll_scratch = h->scratch_ll;
            a.sync = h->team_sync;
            a.prof = h->team_prof;
            CK(h, cudaMemsetAsync(h->team_sync, 0, team_sync_words(h->res_plan) * sizeof(unsigned int), h->stream));
            if (instrument) CK(h, cudaEventRecord(ev.first, h->stream));
            CK(h, launch_team_block(h->res_plan, a, h->stream));
            h->launches += 1;
        } else {
            ObsBlockArgs a{};
            a.d = h->d;
            a.d.dsum_cur = a.d.dsum_prop = nullptr;
            a.descs = sl.d_descs; a.n_steps = n_steps;
            a.obs = h->obs_dev; a.n_obs = h->n_obs_local;
            a.go = h->blk_go; a.counter = h->blk_counter;
            if (instrument) CK(h, cudaEventRecord(ev.first, h->stream));
            CK(h, launch_obs_block(h->obsblk_plan, a, h->stream));
            h->launches += 1;
        }
        if (instrument) {
            CK(h, cudaEventRecord(ev.second, h->stream));
            h->ev_pending.push_back(ev);
        }
        h->grad_valid = kind_is_mala(kinds[n_steps - 1]);
        h->dc_valid = false;
    } else if (!use_graph) {
        CK(h, cudaMemcpyAsync(sl.d_descs, sl.h_descs, sizeof(StepDesc) * n_steps,
                              cudaMemcpyHostToDevice, h->stream));
        if ((rc = enqueue_steps(h, sl.d_descs, kinds.data(), n_steps, instrument, h->grad_valid, h->dc_valid))) return rc;
    } else {
        // the kernel sequence depends on the kinds of the block's updates (and on whether the
        // current-state gradient is fresh), not on which update each element names
        const long long key = (long long)((hash << 1) | (unsigned long long)si);
        auto it = h->graphs.find(key);
        if (it == h->graphs.end()) {
            const int64_t launches_before = h->launches;
            bool gv = h->grad_valid, dc = h->dc_valid;
            cudaGraph_t g = nullptr;
            CK(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
            cudaError_t e1 = cudaMemcpyAsync(sl.d_descs, sl.h_descs, sizeof(StepDesc) * n_steps,
                                             cudaMemcpyHostToDevice, h->stream);
            int32_t rc2 = e1 == cudaSuccess ? enqueue_steps(h, sl.d_descs, kinds.data(), n_steps, false, gv, dc) : EXTMCMC_ECUDA;
            cudaError_t e2 = cudaStreamEndCapture(h->stream, &g);
            h->graph_launches[key] = h->launches - launches_before;
            h->launches = launches_before;
            if (rc2 || e2 != cudaSuccess || !g) {
                if (g) cudaGraphDestroy(g);
                return fail(h, EXTMCMC_ECUDA, "CUDA graph capture failed: " + h->err);
            }
            cudaGraphExec_t ge = nullptr;
            cudaError_t e3 = cudaGraphInstantiate(&ge, g, 0);
            cudaGraphDestroy(g);
            if (e3 != cudaSuccess)
                return fail(h, EXTMCMC_ECUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e3));
            it = h->graphs.emplace(key, ge).first;
        }
        CK(h, cudaGraphLaunch(it->second, h->stream));
        h->launches += h->graph_launches[key];
        for (int s = 0; s < n_steps; ++s) step_advance(h->dcache, kinds[s], h->grad_valid, h->dc_valid);
    }
    CK(h, cudaEventRecord(sl.done, h->stream));
    sl.in_flight = true;
    h->seq_next += n_steps;
    h->xseq_next += n_steps;
    return EXTMCMC_OK;
}

}  // namespace

// =====================================================================================
extern "C" {

int32_t extmcmc_abi_version(void) { return EXTMCMC_ABI_VERSION; }

const char *extmcmc_last_error(extmcmc_t h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int32_t extmcmc_create(const extmcmc_config_t *cfg, extmcmc_t *out) {
    if (!cfg || !out) return fail(nullptr, EXTMCMC_EINVAL, "null argument");
    *out = nullptr;
    if (cfg->abi_version != EXTMCMC_ABI_VERSION) return fail(nullptr, EXTMCMC_EINVAL, "ABI version mismatch");
    if (cfg->n_chains < 1 || cfg->n_params < 1 || cfg->n_updates < 1 || cfg->history_window < 1)
        return fail(nullptr, EXTMCMC_EINVAL, "n_chains, n_params, n_updates, history_window must be >= 1");
    if (cfg->n_updates > 65535) return fail(nullptr, EXTMCMC_EINVAL, "n_updates must be < 65536");
    switch (cfg->law) {
    case EXTMCMC_LAW_GSN_IID_1D:
        if (cfg->obs_dim != 1 || cfg->n_params != 2)
            return fail(nullptr, EXTMCMC_EINVAL, "GSN_IID_1D needs obs_dim = 1, n_params = 2");
        break;
    case EXTMCMC_LAW_GSN_MV:
        if (cfg->obs_dim < 2 || cfg->obs_dim > kMaxObsDim)
            return fail(nullptr, EXTMCMC_EUNSUPPORTED, "GSN_MV on the GPU path needs 2 <= obs_dim <= 16 (d = 1: GSN_IID_1D)");
        if (cfg->n_params != cfg->obs_dim * (cfg->obs_dim + 1))
            return fail(nullptr, EXTMCMC_EINVAL, "GSN_MV needs n_params = d (d + 1)");
        break;
    case EXTMCMC_LAW_LOGISTIC:
        if (cfg->obs_dim != cfg->n_params || cfg->obs_dim < 1 || logistic_padded_dim(cfg->obs_dim) == 0)
            return fail(nullptr, EXTMCMC_EUNSUPPORTED, "LOGISTIC needs obs_dim = n_params = d with 1 <= d <= 256");
        break;
    case EXTMCMC_LAW_HIER_NORMAL:
        if (cfg->obs_dim != 1 || cfg->n_params < 3)
            return fail(nullptr, EXTMCMC_EINVAL, "HIER_NORMAL needs obs_dim = 1 and n_params = G + 2 >= 3");
        break;
    case EXTMCMC_LAW_USER:
        if (cfg->obs_dim < 1 || cfg->obs_dim > kUserMaxObsDim || cfg->n_params > kUserMaxParams)
            return fail(nullptr, EXTMCMC_EUNSUPPORTED, "USER needs 1 <= obs_dim <= 64 and 1 <= n_params <= 64");
        // When this is built, only rank 0 adds a law's logpdf_theta (EXTMCMC_USER_THETA_TERM): the per-chain
        // sums of all ranks are added up, and the term belongs to the whole likelihood once.
        if (cfg->shard_mode == EXTMCMC_SHARD_OBS && cfg->world_size > 1)
            return fail(nullptr, EXTMCMC_EUNSUPPORTED, "user laws are not implemented under EXTMCMC_SHARD_OBS with several ranks");
        break;
    default:
        // the reference's convention for a missing method: error("... not implemented")
        return fail(nullptr, EXTMCMC_EUNSUPPORTED, "target law not implemented on the GPU path");
    }
    if (cfg->stats_mode < 0 || cfg->stats_mode > 2) return fail(nullptr, EXTMCMC_EINVAL, "bad stats_mode");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, EXTMCMC_ECUDA,
                    std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count = 0"));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, EXTMCMC_EINVAL, "bad device ordinal");

    extmcmc_handle *h = new extmcmc_handle();
    h->cfg = *cfg;
    auto bail = [&](int32_t rc) { g_create_error = h->err; extmcmc_destroy(h); return rc; };
#define CKC(call)                                                                        \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                 \
            return bail(e_ == cudaErrorMemoryAllocation ? EXTMCMC_EOOM : EXTMCMC_ECUDA); \
        }                                                                                \
    } while (0)
    CKC(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CKC(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) {
        h->err = "libextmcmc_cuda is built for sm_100a (B200) only; found sm_" +
                 std::to_string(prop.major) + std::to_string(prop.minor);
        return bail(EXTMCMC_EUNSUPPORTED);
    }
    h->num_sms = prop.multiProcessorCount;
    h->l2_bytes = (size_t)prop.l2CacheSize;
    CKC(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CKC(cudaEventCreateWithFlags(&h->fetch_ready, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&h->fetch_done, cudaEventDisableTiming));
    CKC(cudaEventCreate(&h->t0));
    CKC(cudaEventCreate(&h->t1));
    for (auto &sl : h->slot) CKC(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    CKC(sweep_gsn1d_init());
    CKC(sweep_logistic_init());
    h->logi_D = cfg->law == EXTMCMC_LAW_LOGISTIC ? logistic_padded_dim(cfg->obs_dim) : 0;

    DevState &d = h->d;
    const int64_t C = cfg->n_chains;
    const int p = cfg->n_params, NU = cfg->n_updates;
    d.C = C; d.gC = C; d.g0 = 0; d.chain_offset = cfg->chain_offset; d.p = p; d.NU = NU;
    d.W = cfg->roll_window > 0 ? cfg->roll_window : 100;
    d.H = cfg->history_window;
    d.law = cfg->law; d.stats_mode = cfg->stats_mode; d.rng_mode = EXTMCMC_RNG_PHILOX;
    d.p_u_max = 1; d.seed = cfg->seed;
    d.obs_dim = cfg->obs_dim;
    d.G = cfg->law == EXTMCMC_LAW_HIER_NORMAL ? cfg->n_params - 2 : 1;
    d.lawc_k = cfg->law == EXTMCMC_LAW_GSN_IID_1D ? 3
             : law_self_finished(cfg->law) ? 1
             : cfg->law == EXTMCMC_LAW_HIER_NORMAL ? d.G
             : cfg->obs_dim + cfg->obs_dim * (cfg->obs_dim + 1) / 2 + 1;
    // the accept kernel reads the finished sum from ssum when another kernel produced it:
    // the NCCL all-reduce under observation sharding, or the logistic sweep's own finalize
    d.use_ssum = ((cfg->shard_mode == EXTMCMC_SHARD_OBS && cfg->world_size > 1) ||
                  law_self_finished(cfg->law)) ? 1 : 0;
    int32_t rc = 0;
    const size_t covn = cfg->stats_mode == 0 ? (size_t)p * p : (cfg->stats_mode == 1 ? (size_t)p : 0);
    if ((rc = dev_alloc(h, &d.theta, (size_t)p * C)) || (rc = dev_alloc(h, &d.ll, (size_t)C)) ||
        (rc = dev_alloc(h, &d.prop_loc, (size_t)kMaxCoords * C)) ||
        (rc = dev_alloc(h, &d.prop_full, (size_t)p * C)) ||
        (rc = dev_alloc(h, &d.lawc, (size_t)d.lawc_k * C)) ||
        (rc = dev_alloc(h, &d.n_used, (size_t)C)) || (rc = dev_alloc(h, &d.ssum, (size_t)C)) ||
        (rc = dev_alloc(h, &d.ll_prop, (size_t)C)) || (rc = dev_alloc(h, &d.grad_cur, (size_t)p * C)) ||
        (rc = dev_alloc(h, &d.grad_prop, (size_t)p * C)) ||
        (rc = dev_alloc(h, &h->goff_dev, (size_t)d.G)) || (rc = dev_alloc(h, &h->glen_dev, (size_t)d.G)) ||
        (rc = dev_alloc(h, &d.mean, (size_t)p * C)) || (rc = dev_alloc(h, &d.cov, covn * C)) ||
        (rc = dev_alloc(h, &d.h_theta, (size_t)d.H * p * C)) ||
        (rc = dev_alloc(h, &d.h_prop, (size_t)d.H * p * C)) ||
        (rc = dev_alloc(h, &d.h_ll, (size_t)d.H * C)) || (rc = dev_alloc(h, &d.h_llp, (size_t)d.H * C)) ||
        (rc = dev_alloc(h, &d.h_acc, (size_t)d.H * C)) || (rc = dev_alloc(h, &d.err_flag, 1)) ||
        (rc = dev_alloc(h, &d.upd, (size_t)NU)) || (rc = dev_alloc(h, &h->scratch_ll, (size_t)C)) ||
        (rc = dev_alloc(h, &h->n_obs_dev, 1)))
        return bail(rc);
    CKC(cudaMemset(d.err_flag, 0, sizeof(int32_t)));
    h->upd_host.assign(NU, DevUpdate{});
    h->upd_set.assign(NU, false);
    h->ra_iter.assign(NU, 0);
    h->acc_tag.assign((size_t)NU * d.W, 0);
    h->haario_M.assign(NU, 0);
    h->lambda.assign(NU, 0.0);
    h->lambda_fn.assign(NU, nullptr);
    h->lambda_user.assign(NU, nullptr);
    if (cfg->law == EXTMCMC_LAW_GSN_MV && (rc = dev_alloc(h, &d.mv_L, (size_t)cfg->obs_dim * cfg->obs_dim * C)))
        return bail(rc);
    {
        // bounded wait for the peers' sums under observation sharding (and for the go-flag of the
        // observation-mapped block kernel): generous, because ordinary host skew (a rank inside a
        // callback, a first-block graph capture) delays a peer's launch, not only a dead rank
        const char *e = getenv("EXTMCMC_P2P_TIMEOUT_MS");
        const double ms = e ? atof(e) : 30000.0;
        d.p2p_timeout_ns = (unsigned long long)((ms > 1.0 ? ms : 1.0) * 1e6);
    }
    *out = h;
    return EXTMCMC_OK;
#undef CKC
}

int32_t extmcmc_destroy(extmcmc_t h) {
    if (!h) return EXTMCMC_OK;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->team_prof) {
        // diagnostics: where the CTAs of the team kernel spent their cycles (mean over CTAs and launches)
        const int n = h->res_plan.n_cta;
        std::vector<long long> pr((size_t)n * 8);
        if (cudaMemcpy(pr.data(), h->team_prof, pr.size() * sizeof(long long), cudaMemcpyDeviceToHost) == cudaSuccess) {
            double s[7] = {0, 0, 0, 0, 0, 0, 0}, runs = 0, mx = 0, mn = 1e300;
            for (int b = 0; b < n; ++b) {
                double tot = 0;
                for (int i = 0; i < 7; ++i) { s[i] += (double)pr[(size_t)b * 8 + i]; tot += (double)pr[(size_t)b * 8 + i]; }
                runs += (double)pr[(size_t)b * 8 + 7];
                if (pr[(size_t)b * 8 + 7]) { const double t = tot / pr[(size_t)b * 8 + 7]; mx = std::max(mx, t); mn = std::min(mn, t); }
            }
            if (runs > 0)
                fprintf(stderr, "[extmcmc team kernel] cycles per launch per CTA: sweep %.0f, barrier-before %.0f, barrier-after %.0f, "
                                "propose %.0f, accept %.0f, cov+sync %.0f, ctx %.0f; total min %.0f max %.0f over CTAs; %d CTAs, ts %d, stages %d\n",
                        s[0] / runs, s[1] / runs, s[2] / runs, s[3] / runs, s[4] / runs, s[5] / runs, s[6] / runs, mn, mx, n,
                        h->res_plan.ts, h->res_plan.stages);
        }
    }
    invalidate_graphs(h);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    for (void *p : h->p2p_opened) cudaIpcCloseMemHandle(p);
    if (h->p2p_region) cudaFree(h->p2p_region);
    for (void *p : h->allocs) cudaFree(p);
    if (h->obs_dev) cudaFree(h->obs_dev);
    if (h->y_dev) cudaFree(h->y_dev);
    user_law_unload(h->ulaw);
    if (h->rp_prop) cudaFree(h->rp_prop);
    if (h->rp_exp) cudaFree(h->rp_exp);
    if (h->flush_buf) cudaFree(h->flush_buf);
    for (auto &sl : h->slot) {
        if (sl.h_descs) cudaFreeHost(sl.h_descs);
        if (sl.d_descs) cudaFree(sl.d_descs);
        if (sl.done) cudaEventDestroy(sl.done);
    }
    for (auto &ev : h->ev_pending) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    for (auto &ev : h->ev_free) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    if (h->t0) cudaEventDestroy(h->t0);
    if (h->t1) cudaEventDestroy(h->t1);
    for (cudaEvent_t e : h->ev_pool) if (e) cudaEventDestroy(e);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    if (h->fetch_ready) cudaEventDestroy(h->fetch_ready);
    if (h->fetch_done) cudaEventDestroy(h->fetch_done);
    if (h->stage) cudaFreeHost(h->stage);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return EXTMCMC_OK;
}

// Device layout of the observations: group g occupies [goff[g], goff[g] + glen[g]) doubles with
// goff even (16-byte units of the sweep's bulk copies) and one spare pair at the end.
static int32_t install_obs(extmcmc_t h, int64_t n_obs, const std::vector<int64_t> &glen) {
    if (h->obs_dev) { cudaFree(h->obs_dev); h->obs_dev = nullptr; }
    const int G = (int)glen.size();
    std::vector<int64_t> goff(G);
    int64_t tot = 0, largest = 0;
    for (int g = 0; g < G; ++g) {
        goff[g] = tot;
        tot += (glen[g] * h->cfg.obs_dim + 1) & ~(int64_t)1;
        largest = std::max(largest, glen[g]);
    }
    const size_t padded = (size_t)tot + 2;
    CK(h, cudaMalloc(&h->obs_dev, padded * sizeof(double)));
    CK(h, cudaMemsetAsync(h->obs_dev, 0, padded * sizeof(double), h->stream));
    CK(h, cudaMemcpyAsync(h->goff_dev, goff.data(), sizeof(int64_t) * G, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaMemcpyAsync(h->glen_dev, glen.data(), sizeof(int64_t) * G, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    h->n_obs_local = n_obs;
    h->n_obs_largest = largest;
    h->plan_valid = false;
    h->n_total_known = false;
    h->grad_valid = false;
    h->dc_valid = false;
    return EXTMCMC_OK;
}

int32_t extmcmc_upload_obs(extmcmc_t h, const double *obs, int64_t n_obs, int32_t obs_dim,
                           const double *y) {
    if (!h) return EXTMCMC_EINVAL;
    if (!obs || n_obs < 1) return fail(h, EXTMCMC_EINVAL, "need at least one observation");
    if (obs_dim != h->cfg.obs_dim) return fail(h, EXTMCMC_EINVAL, "obs_dim differs from the configuration");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->cfg.law == EXTMCMC_LAW_LOGISTIC) {
        // X -> [n_pad][D] (zero rows up to a multiple of 16, zero columns up to D), y -> [n_pad]
        if (!y) return fail(h, EXTMCMC_EINVAL, "LOGISTIC needs the responses y");
        const int D = h->logi_D;
        const size_t n_pad = ((size_t)n_obs + 15) & ~(size_t)15;
        if (h->obs_dev) { cudaFree(h->obs_dev); h->obs_dev = nullptr; }
        if (h->y_dev) { cudaFree(h->y_dev); h->y_dev = nullptr; }
        CK(h, cudaMalloc(&h->obs_dev, n_pad * D * sizeof(double)));
        CK(h, cudaMalloc(&h->y_dev, n_pad * sizeof(double)));
        CK(h, cudaMemsetAsync(h->obs_dev, 0, n_pad * D * sizeof(double), h->stream));
        CK(h, cudaMemsetAsync(h->y_dev, 0, n_pad * sizeof(double), h->stream));
        CK(h, cudaMemcpy2DAsync(h->obs_dev, (size_t)D * 8, obs, (size_t)obs_dim * 8, (size_t)obs_dim * 8,
                                (size_t)n_obs, cudaMemcpyHostToDevice, h->stream));
        CK(h, cudaMemcpyAsync(h->y_dev, y, (size_t)n_obs * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        h->n_obs_local = n_obs;
        h->n_obs_largest = n_obs;
        h->plan_valid = false;
        h->n_total_known = false;
        h->grad_valid = false;
        h->dc_valid = false;
        return EXTMCMC_OK;
    }
    if (h->cfg.law == EXTMCMC_LAW_USER) {
        // rows [n_pad][D], n_pad even: every tile of the sweep is a whole number of 16-byte units
        if (y) return fail(h, EXTMCMC_EINVAL, "USER takes no y: responses and covariates are columns of the rows");
        const size_t n_pad = ((size_t)n_obs + 1) & ~(size_t)1, nd = (size_t)n_obs * obs_dim;
        if (h->obs_dev) { cudaFree(h->obs_dev); h->obs_dev = nullptr; }
        CK(h, cudaMalloc(&h->obs_dev, n_pad * obs_dim * sizeof(double)));
        CK(h, cudaMemsetAsync(h->obs_dev, 0, n_pad * obs_dim * sizeof(double), h->stream));
        CK(h, cudaMemcpyAsync(h->obs_dev, obs, nd * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        h->n_obs_local = n_obs;
        h->n_obs_largest = n_obs;
        h->plan_valid = false;
        h->n_total_known = false;
        h->grad_valid = false;
        h->dc_valid = false;
        return EXTMCMC_OK;
    }
    std::vector<int64_t> glen(h->d.G, 0);
    if (h->cfg.law == EXTMCMC_LAW_HIER_NORMAL) {
        // y[i] = group index of observation i (0-based), non-decreasing
        if (!y) return fail(h, EXTMCMC_EINVAL, "HIER_NORMAL needs the group index of every observation in y");
        int64_t prev = 0;
        for (int64_t i = 0; i < n_obs; ++i) {
            const int64_t g = (int64_t)y[i];
            if (g < prev || g >= h->d.G || (double)g != y[i])
                return fail(h, EXTMCMC_EINVAL, "group indices must be integers in [0, G), sorted ascending");
            prev = g;
            ++glen[g];
        }
    } else {
        glen[0] = n_obs;
    }
    int32_t rc = install_obs(h, n_obs, glen);
    if (rc) return rc;
    int64_t src = 0, dst = 0;
    for (int g = 0; g < h->d.G; ++g) {
        const int64_t nd = glen[g] * obs_dim;
        if (nd) CK(h, cudaMemcpyAsync(h->obs_dev + dst, obs + src, (size_t)nd * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        src += nd;
        dst += (nd + 1) & ~(int64_t)1;
    }
    CK(h, cudaStreamSynchronize(h->stream));
    return EXTMCMC_OK;
}

int32_t extmcmc_generate_obs_normal(extmcmc_t h, int64_t first, int64_t n_obs, double mean, double sd,
                                    uint64_t seed) {
    if (!h) return EXTMCMC_EINVAL;
    if (n_obs < 1 || first < 0 || !(sd > 0.0)) return fail(h, EXTMCMC_EINVAL, "bad generate_obs arguments");
    if (h->cfg.law != EXTMCMC_LAW_GSN_IID_1D) return fail(h, EXTMCMC_EUNSUPPORTED, "generate_obs_normal needs the GSN_IID_1D law");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    int32_t rc = install_obs(h, n_obs, std::vector<int64_t>{n_obs});
    if (rc) return rc;
    launch_generate_obs_normal(h->obs_dev, first, n_obs, mean, sd, seed, h->num_sms, h->stream);
    h->launches += 1;
    CK(h, cudaGetLastError());
    CK(h, cudaStreamSynchronize(h->stream));
    return EXTMCMC_OK;
}

// Per-chain SoA scratch of the Gaussian walks, Haario registration and MvNormal priors: three
// columns of n doubles per chain (step_device.cuh).  Grown on demand, never shrunk.
static int32_t ensure_gw_scratch(extmcmc_t h, int n) {
    if (n <= h->d.gw_n) return EXTMCMC_OK;
    CK(h, cudaStreamSynchronize(h->stream));
    double *p = nullptr;
    int32_t rc = dev_alloc(h, &p, (size_t)3 * n * h->d.C);
    if (rc) return rc;
    h->d.gw = p;
    h->d.gw_n = n;
    invalidate_graphs(h);
    return EXTMCMC_OK;
}

int32_t extmcmc_set_update(extmcmc_t h, int32_t u, const extmcmc_update_t *upd) {
    if (!h || !upd) return EXTMCMC_EINVAL;
    if (u < 0 || u >= h->cfg.n_updates) return fail(h, EXTMCMC_EINVAL, "update index out of range");
    // ---- validation first: a failed call leaves the update as it was -----------------------------
    const bool gauss = upd->kernel == EXTMCMC_KERNEL_RW_GAUSS || upd->kernel == EXTMCMC_KERNEL_RW_GAUSS_MIX;
    const bool mala = upd->kernel == EXTMCMC_KERNEL_MALA;
    const bool mix = upd->kernel == EXTMCMC_KERNEL_RW_GAUSS_MIX;
    const bool haario = upd->adapt.kind == EXTMCMC_ADAPT_HAARIO;
    if (upd->kernel != EXTMCMC_KERNEL_RW_UNIFORM && !gauss && !mala)
        return fail(h, EXTMCMC_EUNSUPPORTED, "transition kernel not implemented on the GPU path");
    if (mala) {
        if (h->cfg.law != EXTMCMC_LAW_GSN_IID_1D && h->cfg.law != EXTMCMC_LAW_HIER_NORMAL &&
            h->cfg.law != EXTMCMC_LAW_LOGISTIC && h->cfg.law != EXTMCMC_LAW_USER)
            return fail(h, EXTMCMC_EUNSUPPORTED, "MALA needs a law with a device gradient (GSN_IID_1D, HIER_NORMAL, LOGISTIC, USER)");
        if (h->cfg.law == EXTMCMC_LAW_USER && h->ulaw.loaded && !h->ulaw.grad)
            return fail(h, EXTMCMC_EUNSUPPORTED, "MALA needs a user law with a gradient (extmcmc_set_user_law with_grad = 1 or 2)");
        if (upd->prior != EXTMCMC_PRIOR_IMPROPER && upd->prior != EXTMCMC_PRIOR_NORMAL)
            return fail(h, EXTMCMC_EUNSUPPORTED, "MALA supports ImproperPrior and Normal priors only");
        if (upd->pos)
            for (int i = 0; i < upd->n_coords; ++i)
                if (upd->pos[i]) return fail(h, EXTMCMC_EUNSUPPORTED, "MALA on positivity-constrained coordinates is not implemented");
    }
    if (upd->prior < EXTMCMC_PRIOR_IMPROPER || upd->prior > EXTMCMC_PRIOR_MVNORMAL)
        return fail(h, EXTMCMC_EUNSUPPORTED, "prior not implemented on the GPU path");
    if (upd->n_coords < 1 || upd->n_coords > (mala ? std::min(h->cfg.n_params, 32768) : kMaxCoords))
        return fail(h, EXTMCMC_EUNSUPPORTED, mala ? "1 <= n_coords <= min(n_params, 32768) for MALA"
                                                  : "1 <= n_coords <= 32 for random-walk updates on the GPU path");
    if (!upd->coords || !upd->step) return fail(h, EXTMCMC_EINVAL, "coords/step missing");
    const int nc = upd->n_coords, nn = nc * nc;
    if (upd->prior == EXTMCMC_PRIOR_PRODUCT) {
        // {K, then per factor: kind, dim, p0, p1}; the dims must tile the update's coordinates
        if (upd->n_prior_params < 1 || !upd->prior_params) return fail(h, EXTMCMC_EINVAL, "ProductPrior parameters missing");
        const int K = (int)upd->prior_params[0];
        if (K < 1 || K > kMaxPriorFactors || upd->n_prior_params != 1 + 4 * K)
            return fail(h, EXTMCMC_EUNSUPPORTED, "ProductPrior: 1 <= factors <= 16");
        int tot = 0;
        for (int k = 0; k < K; ++k) {
            const int kind = (int)upd->prior_params[1 + 4 * k], dim = (int)upd->prior_params[2 + 4 * k];
            if (kind < EXTMCMC_PRIOR_IMPROPER || kind > EXTMCMC_PRIOR_CAUCHY || kind == EXTMCMC_PRIOR_PRODUCT || dim < 1)
                return fail(h, EXTMCMC_EUNSUPPORTED, "ProductPrior factor not implemented on the GPU path");
            tot += dim;
        }
        if (tot != nc) return fail(h, EXTMCMC_EINVAL, "ProductPrior dims must add up to length(coords)");
    } else if (upd->prior == EXTMCMC_PRIOR_MVNORMAL) {
        if (upd->n_prior_params != nc + nn || !upd->prior_params)
            return fail(h, EXTMCMC_EINVAL, "MvNormal prior needs {mu[p_u], L[p_u * p_u]}");
        for (int i = 0; i < nc; ++i)
            if (!(upd->prior_params[nc + i + i * nc] > 0.0))
                return fail(h, EXTMCMC_EINVAL, "MvNormal prior: the Cholesky factor must have a positive diagonal");
    } else {
        if (upd->n_prior_params > kMaxPriorParams || (upd->n_prior_params > 0 && !upd->prior_params))
            return fail(h, EXTMCMC_EINVAL, "bad prior parameters");
        // parameters each StandardPrior family reads
        const int pk = upd->prior;
        const int need = (pk == EXTMCMC_PRIOR_IMPROPER || pk == EXTMCMC_PRIOR_IMPROPER_POS) ? 0
                       : pk == EXTMCMC_PRIOR_EXPONENTIAL ? 1 : 2;
        if (upd->n_prior_params < need) return fail(h, EXTMCMC_EINVAL, "prior parameters missing");
    }
    // readjust! exists only for (UniformRandomWalk, AdaptationUnifRW) and
    // (GaussianRandomWalkMix, HaarioTypeAdaptation): adaptation.jl:273,422
    if (!(upd->adapt.kind == EXTMCMC_ADAPT_NONE ||
          (upd->adapt.kind == EXTMCMC_ADAPT_MALA && mala) ||
          (upd->adapt.kind == EXTMCMC_ADAPT_UNIF_RW && upd->kernel == EXTMCMC_KERNEL_RW_UNIFORM) ||
          (upd->adapt.kind == EXTMCMC_ADAPT_HAARIO && mix)))
        return fail(h, EXTMCMC_EUNSUPPORTED, "adaptation not implemented for this transition kernel");
    if (upd->adapt.kind != EXTMCMC_ADAPT_NONE && upd->adapt.adapt_every_k_steps < 1)
        return fail(h, EXTMCMC_EINVAL, "adapt_every_k_steps must be >= 1");
    for (int i = 0; i < nc; ++i) {
        if (upd->coords[i] < 0 || upd->coords[i] >= h->cfg.n_params)
            return fail(h, EXTMCMC_EINVAL, "coordinate out of range");
        if (!gauss && !mala && !(upd->step[i] > 0.0))  // UniformRandomWalk: @assert all(eps .> 0.0), random_walk.jl:50
            return fail(h, EXTMCMC_EINVAL, "eps must be > 0");
    }
    if (mix && !(upd->step[2 * nn] >= 0.0 && upd->step[2 * nn] <= 1.0))   // @assert 0 <= lambda <= 1, random_walk.jl:199
        return fail(h, EXTMCMC_EINVAL, "lambda must be in [0, 1]");
    if (mala && !(upd->step[0] > 0.0)) return fail(h, EXTMCMC_EINVAL, "MALA step tau must be > 0");
    const bool fresh = !h->upd_set[u];
    {
        const DevUpdate &cur = h->upd_host[u];
        if (!fresh && cur.n_coords != nc) return fail(h, EXTMCMC_EINVAL, "cannot change n_coords of an update");
        if (!fresh && ((mix && !cur.sigB) || (gauss && !cur.sigA) || (haario && !cur.hmean) ||
                       (upd->prior == EXTMCMC_PRIOR_MVNORMAL && !cur.prior_dev)))
            return fail(h, EXTMCMC_EINVAL, "cannot change the kernel or prior family of an update");
    }

    // ---- build the new entry in a copy; it replaces the old one only when everything succeeded ----
    CK(h, cudaSetDevice(h->cfg.device));
    const int64_t C = h->d.C;
    const int W = h->d.W;
    DevUpdate t = h->upd_host[u];
    t.kernel = upd->kernel; t.n_coords = nc; t.prior = upd->prior;
    t.adapt_kind = upd->adapt.kind;
    for (int i = 0; i < nc && i < kMaxCoords; ++i) {
        t.coords[i] = upd->coords[i];
        t.pos[i] = upd->pos ? upd->pos[i] : 0;
    }
    const bool mvn = upd->prior == EXTMCMC_PRIOR_MVNORMAL;
    for (int i = 0; i < kMaxPriorParams; ++i)
        t.prior_params[i] = (!mvn && i < upd->n_prior_params) ? upd->prior_params[i] : 0.0;
    t.adapt_every_k = upd->adapt.adapt_every_k_steps;
    t.target = upd->adapt.target_accpt_rate; t.scale = upd->adapt.scale;
    t.vmin = upd->adapt.min; t.vmax = upd->adapt.max; t.offset = upd->adapt.offset;
    int32_t rc = 0;
    if (fresh) {
        double *pd = nullptr;
        if ((rc = dev_alloc(h, &t.coords_dev, (size_t)nc)) ||
            (rc = dev_alloc(h, &t.eps, (size_t)nc * C)) ||
            (rc = dev_alloc(h, &t.adapt_prop, (size_t)C)) || (rc = dev_alloc(h, &t.adapt_acc, (size_t)C)) ||
            (rc = dev_alloc(h, &t.tot_prop, (size_t)C)) || (rc = dev_alloc(h, &t.tot_acc, (size_t)C)) ||
            (rc = dev_alloc(h, &t.ra_val, (size_t)C)) || (rc = dev_alloc(h, &t.acc_ring, (size_t)W * C)))
            return rc;
        if (gauss && ((rc = dev_alloc(h, &t.sigA, (size_t)nn)) || (rc = dev_alloc(h, &t.LA, (size_t)nn)))) return rc;
        if (mix && ((rc = dev_alloc(h, &t.sigB, (size_t)nn * C)) || (rc = dev_alloc(h, &t.LB, (size_t)nn * C)))) return rc;
        if (haario && ((rc = dev_alloc(h, &t.hmean, (size_t)nc * C)) || (rc = dev_alloc(h, &t.hcov, (size_t)nn * C)))) return rc;
        if (mvn) { if ((rc = dev_alloc(h, &pd, (size_t)(nc + nn)))) return rc; t.prior_dev = pd; }
    }
    if ((gauss || haario || mvn) && (rc = ensure_gw_scratch(h, nc))) return rc;
    CK(h, cudaStreamSynchronize(h->stream));
    CK(h, cudaMemcpy(t.coords_dev, upd->coords, sizeof(int32_t) * nc, cudaMemcpyHostToDevice));
    if (mvn) CK(h, cudaMemcpy(const_cast<double *>(t.prior_dev), upd->prior_params, sizeof(double) * (nc + nn), cudaMemcpyHostToDevice));
    if (mala) {
        std::vector<double> tau0((size_t)C, upd->step[0]);   // one step size tau per chain
        CK(h, cudaMemcpy(t.eps, tau0.data(), tau0.size() * sizeof(double), cudaMemcpyHostToDevice));
    } else if (!gauss) {
        // broadcast the initial step size to every chain
        std::vector<double> eps0((size_t)nc * C);
        for (int i = 0; i < nc; ++i) std::fill_n(eps0.begin() + (size_t)i * C, C, upd->step[i]);
        CK(h, cudaMemcpy(t.eps, eps0.data(), eps0.size() * sizeof(double), cudaMemcpyHostToDevice));
    } else {
        CK(h, cudaMemcpy(t.sigA, upd->step, sizeof(double) * nn, cudaMemcpyHostToDevice));
        launch_chol_factor(t.sigA, t.LA, nc, 1, 1, h->stream);          // L_A, once: Sigma_A never changes
        if (mix) {
            std::vector<double> sb((size_t)nn * C);
            for (int k = 0; k < nn; ++k) std::fill_n(sb.begin() + (size_t)k * C, C, upd->step[nn + k]);
            CK(h, cudaMemcpy(t.sigB, sb.data(), sb.size() * sizeof(double), cudaMemcpyHostToDevice));
            launch_chol_factor(t.sigB, t.LB, nc, C, C, h->stream);      // L_B per chain (rewritten at every readjust!)
        }
        CK(h, cudaGetLastError());
        CK(h, cudaStreamSynchronize(h->stream));
        if (haario) {
            CK(h, cudaMemset(t.hmean, 0, sizeof(double) * nc * C));
            CK(h, cudaMemset(t.hcov, 0, sizeof(double) * nn * C));
        }
    }
    CK(h, cudaMemset(t.adapt_prop, 0, sizeof(int32_t) * C));
    CK(h, cudaMemset(t.adapt_acc, 0, sizeof(int32_t) * C));
    CK(h, cudaMemset(t.tot_prop, 0, sizeof(int64_t) * C));
    CK(h, cudaMemset(t.tot_acc, 0, sizeof(int64_t) * C));
    CK(h, cudaMemset(t.ra_val, 0, sizeof(double) * C));
    CK(h, cudaMemset(t.acc_ring, 0, (size_t)W * C));
    h->upd_host[u] = t;
    h->lambda[u] = mix ? upd->step[2 * nn] : 0.0;
    h->haario_M[u] = 0;
    h->upd_set[u] = true;
    h->upd_dirty = true;
    h->blk_planned = false;
    int nh = 0;
    h->any_mala = false;
    for (int v = 0; v < h->cfg.n_updates; ++v) {
        if (h->upd_set[v] && h->upd_host[v].kernel == EXTMCMC_KERNEL_MALA) h->any_mala = true;
        if (h->upd_set[v] && h->upd_host[v].adapt_kind == EXTMCMC_ADAPT_HAARIO) ++nh;
    }
    if (nh != h->d.n_haario) { h->d.n_haario = nh; invalidate_graphs(h); }
    // the compact step-kernel instantiations apply when every update is plain (step_device.cuh, SpecLean)
    static const bool lean_on = [] { const char *e = getenv("EXTMCMC_LEAN"); return !e || atoi(e) != 0; }();
    int lean = lean_on ? 1 : 0;
    for (int v = 0; v < h->cfg.n_updates; ++v) {
        if (!h->upd_set[v]) continue;
        const DevUpdate &w = h->upd_host[v];
        if ((w.kernel != EXTMCMC_KERNEL_RW_UNIFORM && w.kernel != EXTMCMC_KERNEL_MALA) || !lean_prior(w.prior) ||
            w.adapt_kind == EXTMCMC_ADAPT_HAARIO)
            lean = 0;
    }
    if (lean != h->d.lean) { h->d.lean = lean; invalidate_graphs(h); }
    return EXTMCMC_OK;
}

int32_t extmcmc_set_seed(extmcmc_t h, uint64_t seed) {
    if (!h) return EXTMCMC_EINVAL;
    h->cfg.seed = seed;
    h->d.seed = seed;
    invalidate_graphs(h);   // the key is baked into the kernel arguments
    return EXTMCMC_OK;
}

int32_t extmcmc_set_lambda_fn(extmcmc_t h, int32_t u, extmcmc_lambda_fn f, void *user) {
    if (!h) return EXTMCMC_EINVAL;
    if (u < 0 || u >= h->cfg.n_updates) return fail(h, EXTMCMC_EINVAL, "update index out of range");
    h->lambda_fn[u] = f;
    h->lambda_user[u] = user;
    return EXTMCMC_OK;
}

int32_t extmcmc_set_state(extmcmc_t h, const double *theta) {
    if (!h || !theta) return EXTMCMC_EINVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    const DevState &d = h->d;
    const int64_t C = d.C;
    CK(h, cudaMemcpy(d.theta, theta, sizeof(double) * d.p * C, cudaMemcpyHostToDevice));
    std::vector<double> ninf((size_t)C, -INFINITY);  // StandardLocalSubworkspace.ll, workspaces.jl:425
    CK(h, cudaMemcpy(d.ll, ninf.data(), sizeof(double) * C, cudaMemcpyHostToDevice));
    CK(h, cudaMemset(d.mean, 0, sizeof(double) * d.p * C));
    const size_t covn = d.stats_mode == 0 ? (size_t)d.p * d.p : (d.stats_mode == 1 ? (size_t)d.p : 0);
    if (covn) CK(h, cudaMemset(d.cov, 0, sizeof(double) * covn * C));
    CK(h, cudaMemset(d.err_flag, 0, sizeof(int32_t)));
    for (int u = 0; u < h->cfg.n_updates; ++u) {
        if (!h->upd_set[u]) continue;
        DevUpdate &t = h->upd_host[u];
        CK(h, cudaMemset(t.adapt_prop, 0, sizeof(int32_t) * C));
        CK(h, cudaMemset(t.adapt_acc, 0, sizeof(int32_t) * C));
        CK(h, cudaMemset(t.tot_prop, 0, sizeof(int64_t) * C));
        CK(h, cudaMemset(t.tot_acc, 0, sizeof(int64_t) * C));
        CK(h, cudaMemset(t.ra_val, 0, sizeof(double) * C));
        CK(h, cudaMemset(t.acc_ring, 0, (size_t)d.W * C));
        if (t.hmean) {
            CK(h, cudaMemset(t.hmean, 0, sizeof(double) * t.n_coords * C));
            CK(h, cudaMemset(t.hcov, 0, sizeof(double) * t.n_coords * t.n_coords * C));
        }
    }
    std::fill(h->haario_M.begin(), h->haario_M.end(), 0);
    h->seq_next = 0;
    h->grad_valid = false;
    h->dc_valid = false;
    if (h->fetch_active) { cudaEventSynchronize(h->fetch_done); h->fetch_active = false; }
    std::fill(h->ra_iter.begin(), h->ra_iter.end(), 0);
    std::fill(h->acc_tag.begin(), h->acc_tag.end(), 0);
    h->state_set = true;
    return EXTMCMC_OK;
}

}  // extern "C"
namespace {
// with_grad of the C ABI -> UserGrad: EXTMCMC_USER_GRAD_FORWARD, or any other non-zero value: hand-written
int user_grad_mode(int32_t with_grad) {
    return with_grad == EXTMCMC_USER_GRAD_FORWARD ? kUserGradForward : with_grad ? kUserGradHand : kUserValue;
}
std::string forward_limit_message(int32_t n_params) {
    return "forward-mode gradients (with_grad = EXTMCMC_USER_GRAD_FORWARD) need 1 <= n_params <= " +
           std::to_string(kUserMaxForwardParams) + " (every parameter-dependent field of the Law holds n_params + 1 "
           "doubles in registers); got n_params = " + std::to_string(n_params) + ": write logpdf_grad (with_grad = 1).  The chunked entry points (extmcmc_set_user_law_chunked, "
           "extmcmc_user_law_check_chunked) take forward-mode laws of up to 64 parameters.";
}
void copy_log(const std::string &msg, char *log, int64_t log_bytes) {
    if (log && log_bytes > 0) {
        const size_t n = std::min(msg.size(), (size_t)log_bytes - 1);
        std::memcpy(log, msg.data(), n);
        log[n] = 0;
    }
}
// The options of every user-law entry point, checked and resolved to a UserGrad mode and the chunk
// width K of forward mode.  chunked: the width comes from `chunk` (the _chunked and _ex entry points);
// otherwise forward mode is the unchunked program and keeps its limit of kUserMaxForwardParams.
int32_t user_law_options(int32_t P, int32_t with_grad, bool chunked, int32_t chunk, int32_t flags, int &mode, int &K,
                         std::string &err) {
    if (flags & ~EXTMCMC_USER_THETA_TERM) {
        err = "unknown user-law flags " + std::to_string(flags) + " (known: EXTMCMC_USER_THETA_TERM = 1)";
        return EXTMCMC_EINVAL;
    }
    mode = user_grad_mode(with_grad);
    K = P;
    if (mode != kUserGradForward) {
        if (chunk == 0) return EXTMCMC_OK;
        err = "chunk must be 0 unless with_grad = EXTMCMC_USER_GRAD_FORWARD; got " + std::to_string(chunk);
        return EXTMCMC_EINVAL;
    }
    if (chunked) return user_law_chunk(P, chunk, K, err);
    if (P <= kUserMaxForwardParams) return EXTMCMC_OK;
    err = forward_limit_message(P);
    return EXTMCMC_EUNSUPPORTED;
}
// every extmcmc_user_law_check* entry point
int32_t user_law_check(const char *source, int32_t n_params, int32_t obs_dim, int32_t with_grad, bool chunked,
                       int32_t chunk, int32_t flags, int32_t *chunk_used, char *log, int64_t log_bytes) {
    if (log && log_bytes > 0) log[0] = 0;
    if (!source) return fail(nullptr, EXTMCMC_EINVAL, "null source");
    if (n_params < 1 || n_params > kUserMaxParams || obs_dim < 1 || obs_dim > kUserMaxObsDim)
        return fail(nullptr, EXTMCMC_EUNSUPPORTED, "user laws need 1 <= n_params <= 64 and 1 <= obs_dim <= 64");
    int mode = kUserValue, K = 0;
    std::string err;
    if (const int32_t rc = user_law_options(n_params, with_grad, chunked, chunk, flags, mode, K, err)) {
        copy_log(err, log, log_bytes);
        return fail(nullptr, rc, err);
    }
    if (chunk_used) *chunk_used = mode == kUserGradForward ? K : 0;
    std::string lg, cubin;
    const int32_t rc = user_law_compile(source, n_params, obs_dim, mode, K, flags, lg, cubin, nullptr);
    copy_log(lg, log, log_bytes);
    if (rc) g_create_error = lg;
    return rc;
}
// every extmcmc_set_user_law* entry point; entry: its name, for the messages
int32_t set_user_law(extmcmc_t h, const char *entry, const char *source, int32_t with_grad, bool chunked,
                     int32_t chunk, int32_t flags) {
    if (!h) return EXTMCMC_EINVAL;
    if (h->cfg.law != EXTMCMC_LAW_USER) return fail(h, EXTMCMC_EINVAL, std::string(entry) + " needs a handle of law EXTMCMC_LAW_USER");
    if (!source) return fail(h, EXTMCMC_EINVAL, "null source");
    int mode = kUserValue, K = 0;
    std::string err;
    if (const int32_t rc = user_law_options(h->cfg.n_params, with_grad, chunked, chunk, flags, mode, K, err))
        return fail(h, rc, err);
    std::string log, cubin;
    uint64_t hash = 0;
    const int32_t rc = user_law_compile(source, h->cfg.n_params, h->cfg.obs_dim, mode, K, flags, log, cubin, &hash);
    if (rc == EXTMCMC_EINVAL) return fail(h, rc, "the user law does not compile:\n" + log);
    if (rc) return fail(h, rc, log);
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));   // no queued launch may still use the old kernels
    invalidate_graphs(h);
    const cudaError_t e = user_law_load(h->ulaw, cubin, h->cfg.n_params, h->cfg.obs_dim, mode, K, hash);
    if (e != cudaSuccess) {
        user_law_unload(h->ulaw);
        return fail(h, EXTMCMC_ECUDA, std::string("loading the user law: ") + cudaGetErrorString(e));
    }
    h->plan_valid = false;
    h->grad_valid = false;
    return EXTMCMC_OK;
}
}  // namespace
extern "C" {

int32_t extmcmc_user_law_check(const char *source, int32_t n_params, int32_t obs_dim, int32_t with_grad,
                               char *log, int64_t log_bytes) {
    return user_law_check(source, n_params, obs_dim, with_grad, false, 0, 0, nullptr, log, log_bytes);
}

int32_t extmcmc_user_law_check_chunked(const char *source, int32_t n_params, int32_t obs_dim, int32_t chunk,
                                       int32_t *chunk_used, char *log, int64_t log_bytes) {
    return user_law_check(source, n_params, obs_dim, EXTMCMC_USER_GRAD_FORWARD, true, chunk, 0, chunk_used, log,
                          log_bytes);
}

int32_t extmcmc_user_law_check_ex(const char *source, int32_t n_params, int32_t obs_dim, int32_t with_grad,
                                  int32_t chunk, int32_t flags, int32_t *chunk_used, char *log, int64_t log_bytes) {
    return user_law_check(source, n_params, obs_dim, with_grad, true, chunk, flags, chunk_used, log, log_bytes);
}

int32_t extmcmc_set_user_law(extmcmc_t h, const char *source, int32_t with_grad) {
    return set_user_law(h, "extmcmc_set_user_law", source, with_grad, false, 0, 0);
}

int32_t extmcmc_set_user_law_chunked(extmcmc_t h, const char *source, int32_t chunk) {
    return set_user_law(h, "extmcmc_set_user_law_chunked", source, EXTMCMC_USER_GRAD_FORWARD, true, chunk, 0);
}

int32_t extmcmc_set_user_law_ex(extmcmc_t h, const char *source, int32_t with_grad, int32_t chunk, int32_t flags) {
    return set_user_law(h, "extmcmc_set_user_law_ex", source, with_grad, true, chunk, flags);
}

// ---- checkpoint / resume ------------------------------------------------------------------------
}  // extern "C"
namespace {
struct CkptHeader {
    uint64_t magic;
    int64_t C, seq_next;
    int32_t abi, p, NU, W, stats_mode, law, grad_valid, pad;
};
constexpr uint64_t kCkptMagic = 0x32544b434d435845ull;   // "EXCMCKT2"

// Visits every piece of the blob in a fixed order: fn(device pointer or nullptr, host pointer or nullptr, bytes).
template <class F>
int32_t ckpt_walk(extmcmc_t h, F fn) {
    const DevState &d = h->d;
    const size_t C = (size_t)d.C, p = (size_t)d.p;
    const size_t covn = d.stats_mode == 0 ? p * p : (d.stats_mode == 1 ? p : 0);
    int32_t rc;
    if ((rc = fn(d.theta, nullptr, 8 * p * C)) || (rc = fn(d.ll, nullptr, 8 * C))) return rc;
    if (d.stats_mode != 2 && ((rc = fn(d.mean, nullptr, 8 * p * C)) || (rc = fn(d.cov, nullptr, 8 * covn * C)))) return rc;
    if ((rc = fn(nullptr, h->ra_iter.data(), 8 * h->ra_iter.size())) || (rc = fn(nullptr, h->acc_tag.data(), 8 * h->acc_tag.size())) ||
        (rc = fn(nullptr, h->haario_M.data(), 8 * h->haario_M.size())) || (rc = fn(nullptr, h->lambda.data(), 8 * h->lambda.size())))
        return rc;
    for (int u = 0; u < h->cfg.n_updates; ++u) {
        const DevUpdate &t = h->upd_host[u];
        const size_t n = (size_t)t.n_coords, nn = n * n;
        const size_t eps_rows = t.kernel == EXTMCMC_KERNEL_MALA ? 1 : n;
        if ((rc = fn(t.eps, nullptr, 8 * eps_rows * C)) || (rc = fn(t.adapt_prop, nullptr, 4 * C)) ||
            (rc = fn(t.adapt_acc, nullptr, 4 * C)) || (rc = fn(t.tot_prop, nullptr, 8 * C)) || (rc = fn(t.tot_acc, nullptr, 8 * C)) ||
            (rc = fn(t.ra_val, nullptr, 8 * C)) || (rc = fn(t.acc_ring, nullptr, (size_t)d.W * C)))
            return rc;
        if (t.sigB && ((rc = fn(t.sigB, nullptr, 8 * nn * C)) || (rc = fn(t.LB, nullptr, 8 * nn * C)))) return rc;
        if (t.hmean && ((rc = fn(t.hmean, nullptr, 8 * n * C)) || (rc = fn(t.hcov, nullptr, 8 * nn * C)))) return rc;
    }
    return EXTMCMC_OK;
}
}  // namespace
extern "C" {

int32_t extmcmc_checkpoint_size(extmcmc_t h, int64_t *bytes_out) {
    if (!h || !bytes_out) return EXTMCMC_EINVAL;
    for (int u = 0; u < h->cfg.n_updates; ++u)
        if (!h->upd_set[u]) return fail(h, EXTMCMC_EINVAL, "update " + std::to_string(u) + " not set");
    if (h->cfg.law == EXTMCMC_LAW_USER && !h->ulaw.loaded) return fail(h, EXTMCMC_EINVAL, "no user law: call extmcmc_set_user_law first");
    size_t tot = sizeof(CkptHeader) + (h->cfg.law == EXTMCMC_LAW_USER ? sizeof(uint64_t) : 0);   // + hash of the law
    ckpt_walk(h, [&](void *, void *, size_t b) { tot += b; return EXTMCMC_OK; });
    *bytes_out = (int64_t)tot;
    return EXTMCMC_OK;
}

int32_t extmcmc_checkpoint_save(extmcmc_t h, void *blob, int64_t bytes) {
    int64_t need = 0;
    int32_t rc = extmcmc_checkpoint_size(h, &need);
    if (rc) return rc;
    if (!blob || bytes < need) return fail(h, EXTMCMC_EINVAL, "checkpoint buffer too small");
    if (!h->state_set) return fail(h, EXTMCMC_EINVAL, "nothing to save: extmcmc_set_state not called");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    CkptHeader hd{kCkptMagic, h->d.C, h->seq_next, EXTMCMC_ABI_VERSION, h->d.p, h->d.NU, h->d.W, h->d.stats_mode, h->d.law,
                  h->grad_valid ? 1 : 0, 0};
    char *out = (char *)blob;
    std::memcpy(out, &hd, sizeof hd);
    out += sizeof hd;
    if (h->cfg.law == EXTMCMC_LAW_USER) { std::memcpy(out, &h->ulaw.hash, sizeof(uint64_t)); out += sizeof(uint64_t); }
    return ckpt_walk(h, [&](void *dev, void *host, size_t b) -> int32_t {
        if (dev) { CK(h, cudaMemcpy(out, dev, b, cudaMemcpyDeviceToHost)); }
        else std::memcpy(out, host, b);
        out += b;
        return EXTMCMC_OK;
    });
}

int32_t extmcmc_checkpoint_load(extmcmc_t h, const void *blob, int64_t bytes) {
    int64_t need = 0;
    int32_t rc = extmcmc_checkpoint_size(h, &need);
    if (rc) return rc;
    if (!blob || bytes < need) return fail(h, EXTMCMC_EINVAL, "checkpoint blob too small for this configuration");
    CkptHeader hd;
    std::memcpy(&hd, blob, sizeof hd);
    if (hd.magic != kCkptMagic || hd.abi != EXTMCMC_ABI_VERSION || hd.C != h->d.C || hd.p != h->d.p || hd.NU != h->d.NU ||
        hd.W != h->d.W || hd.stats_mode != h->d.stats_mode || hd.law != h->d.law)
        return fail(h, EXTMCMC_EINVAL, "checkpoint does not match this handle (chains, parameters, updates, windows, law)");
    const char *in = (const char *)blob + sizeof hd;
    if (h->cfg.law == EXTMCMC_LAW_USER) {
        uint64_t hash;
        std::memcpy(&hash, in, sizeof hash);
        if (hash != h->ulaw.hash) return fail(h, EXTMCMC_EINVAL, "checkpoint was written under another user law");
        in += sizeof hash;
    }
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    rc = ckpt_walk(h, [&](void *dev, void *host, size_t b) -> int32_t {
        if (dev) { CK(h, cudaMemcpy(dev, in, b, cudaMemcpyHostToDevice)); }
        else std::memcpy(host, in, b);
        in += b;
        return EXTMCMC_OK;
    });
    if (rc) return rc;
    h->seq_next = hd.seq_next;
    h->dc_valid = false;
    h->grad_valid = false;          // (the gradient buffers are not part of the blob: recomputed on demand)
    h->state_set = true;
    h->fetch_active = false;
    CK(h, cudaMemset(h->d.err_flag, 0, sizeof(int32_t)));
    return EXTMCMC_OK;
}

int32_t extmcmc_comm_unique_id(uint8_t id_out[128]) {
    std::string err;
    if (!id_out) return EXTMCMC_EINVAL;
    if (!g_nccl.load(err)) return fail(nullptr, EXTMCMC_ENCCL, err);
    ncclUniqueId id;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) return fail(nullptr, EXTMCMC_ENCCL, "ncclGetUniqueId failed");
    std::memcpy(id_out, &id, 128);
    return EXTMCMC_OK;
}

int32_t extmcmc_comm_init(extmcmc_t h, const uint8_t id_in[128]) {
    if (!h || !id_in) return EXTMCMC_EINVAL;
    if (h->comm) return fail(h, EXTMCMC_EINVAL, "communicator already initialised");
    if (!g_nccl.load(h->err)) return EXTMCMC_ENCCL;
    CK(h, cudaSetDevice(h->cfg.device));
    ncclUniqueId id;
    std::memcpy(&id, id_in, 128);
    NK(h, g_nccl.CommInitRank(&h->comm, h->cfg.world_size, id, h->cfg.rank));
    h->n_total_known = false;
    return EXTMCMC_OK;
}

static size_t p2p_region_bytes(extmcmc_t h) {
    const size_t W = (size_t)h->cfg.world_size;
    return 2 * W * (size_t)h->d.C * 2 * sizeof(unsigned long long);   // rx[2][W][C] cells of two tagged words
}

int32_t extmcmc_p2p_export(extmcmc_t h, uint8_t handle_out[64]) {
    if (!h || !handle_out) return EXTMCMC_EINVAL;
    if (!obs_sharded(h)) return fail(h, EXTMCMC_EINVAL, "peer exchange is for EXTMCMC_SHARD_OBS with world_size > 1");
    if (h->cfg.law != EXTMCMC_LAW_GSN_IID_1D && h->cfg.law != EXTMCMC_LAW_GSN_MV)
        return fail(h, EXTMCMC_EUNSUPPORTED, "peer exchange is implemented for the Gaussian laws");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    CK(h, cudaSetDevice(h->cfg.device));
    if (!h->p2p_region) {
        CK(h, cudaMalloc(&h->p2p_region, p2p_region_bytes(h)));
        CK(h, cudaMemset(h->p2p_region, 0, p2p_region_bytes(h)));
    }
    cudaIpcMemHandle_t hd;
    CK(h, cudaIpcGetMemHandle(&hd, h->p2p_region));
    std::memcpy(handle_out, &hd, 64);
    return EXTMCMC_OK;
}

int32_t extmcmc_p2p_import(extmcmc_t h, const uint8_t *handles) {
    if (!h || !handles) return EXTMCMC_EINVAL;
    if (!h->p2p_region) return fail(h, EXTMCMC_EINVAL, "call extmcmc_p2p_export first");
    CK(h, cudaSetDevice(h->cfg.device));
    const int W = h->cfg.world_size;
    std::vector<unsigned long long *> rx(W);
    for (int q = 0; q < W; ++q) {
        void *base = nullptr;
        if (q == h->cfg.rank) {
            base = h->p2p_region;
        } else {
            cudaIpcMemHandle_t hd;
            std::memcpy(&hd, handles + 64 * (size_t)q, 64);
            CK(h, cudaIpcOpenMemHandle(&base, hd, cudaIpcMemLazyEnablePeerAccess));
            h->p2p_opened.push_back(base);
        }
        rx[q] = (unsigned long long *)base;
    }
    int32_t rc;
    if ((rc = dev_alloc(h, &h->d.peer_rx, (size_t)W))) return rc;
    CK(h, cudaMemcpy(h->d.peer_rx, rx.data(), sizeof(unsigned long long *) * W, cudaMemcpyHostToDevice));
    h->d.my_rx = rx[h->cfg.rank];
    h->d.rank = h->cfg.rank;
    h->d.world = W;
    h->d.p2p = 1;
    invalidate_graphs(h);
    return EXTMCMC_OK;
}

int32_t extmcmc_run_block(extmcmc_t h, const extmcmc_step_t *steps, int32_t n_steps) {
    return run_block_impl(h, steps, n_steps, EXTMCMC_RNG_PHILOX, 0, nullptr, nullptr);
}

int32_t extmcmc_run_block_replay(extmcmc_t h, const extmcmc_step_t *steps, int32_t n_steps,
                                 int32_t p_u_max, const double *proposals, const double *exp_draws) {
    return run_block_impl(h, steps, n_steps, EXTMCMC_RNG_REPLAY, p_u_max, proposals, exp_draws);
}

int32_t extmcmc_sync(extmcmc_t h) {
    if (!h) return EXTMCMC_EINVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    int32_t rc = collect_events(h);
    if (rc) return rc;
    int32_t flag = 0;
    CK(h, cudaMemcpy(&flag, h->d.err_flag, sizeof flag, cudaMemcpyDeviceToHost));
    if (flag == 2)   // sticky until extmcmc_set_state: nothing has been committed since the failed exchange
        return fail(h, EXTMCMC_ENCCL, "peer exchange timed out: a rank did not deliver its partial sums; "
                                      "no step has been committed since (extmcmc_set_state to start over)");
    if (flag == 3)
        return fail(h, EXTMCMC_ECUDA, "a persistent block kernel timed out waiting for its own CTAs (EXTMCMC_P2P_TIMEOUT_MS); "
                                      "the chain state is undefined (extmcmc_set_state to start over)");
    if (flag) {
        CK(h, cudaMemset(h->d.err_flag, 0, sizeof flag));
        return fail(h, EXTMCMC_EDOMAIN,
                    "a chain proposed parameters outside the law's domain (e.g. variance <= 0); "
                    "the proposal was rejected");
    }
    return EXTMCMC_OK;
}

int32_t extmcmc_get_state(extmcmc_t h, double *theta, double *ll) {
    if (!h) return EXTMCMC_EINVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    if (theta) CK(h, cudaMemcpy(theta, h->d.theta, sizeof(double) * h->d.p * h->d.C, cudaMemcpyDeviceToHost));
    if (ll) CK(h, cudaMemcpy(ll, h->d.ll, sizeof(double) * h->d.C, cudaMemcpyDeviceToHost));
    return EXTMCMC_OK;
}

int32_t extmcmc_get_history(extmcmc_t h, int64_t seq_lo, int64_t seq_hi, double *theta,
                            double *theta_prop, double *ll, double *ll_prop, uint8_t *accepted) {
    if (!h) return EXTMCMC_EINVAL;
    if (seq_lo < 0 || seq_hi < seq_lo || seq_hi > h->seq_next) return fail(h, EXTMCMC_EINVAL, "bad history range");
    if (seq_lo < h->seq_next - h->d.H) return fail(h, EXTMCMC_ESTALE, "history rows already overwritten");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    const DevState &d = h->d;
    const int64_t C = d.C, H = d.H;
    int64_t row = 0;
    for (int64_t s = seq_lo; s < seq_hi;) {
        const int64_t slot = s % H;
        const int64_t n = std::min<int64_t>(seq_hi - s, H - slot);  // contiguous run in the ring
        const size_t rp = (size_t)d.p * C;
        if (theta) CK(h, cudaMemcpy(theta + row * rp, d.h_theta + slot * rp, sizeof(double) * n * rp, cudaMemcpyDeviceToHost));
        if (theta_prop) CK(h, cudaMemcpy(theta_prop + row * rp, d.h_prop + slot * rp, sizeof(double) * n * rp, cudaMemcpyDeviceToHost));
        if (ll) CK(h, cudaMemcpy(ll + row * C, d.h_ll + slot * C, sizeof(double) * n * C, cudaMemcpyDeviceToHost));
        if (ll_prop) CK(h, cudaMemcpy(ll_prop + row * C, d.h_llp + slot * C, sizeof(double) * n * C, cudaMemcpyDeviceToHost));
        if (accepted) CK(h, cudaMemcpy(accepted + row * C, d.h_acc + slot * C, (size_t)n * C, cudaMemcpyDeviceToHost));
        s += n;
        row += n;
    }
    return EXTMCMC_OK;
}

// rows [lo, hi) of a ring array with row_bytes per row -> dst (contiguous), on stream st
static int32_t copy_ring_rows(extmcmc_t h, void *dst, const void *ring, size_t row_bytes, int64_t lo,
                              int64_t hi, cudaStream_t st) {
    const int64_t H = h->d.H;
    int64_t row = 0;
    for (int64_t s = lo; s < hi;) {
        const int64_t slot = s % H;
        const int64_t n = std::min<int64_t>(hi - s, H - slot);
        CK(h, cudaMemcpyAsync((char *)dst + row * row_bytes, (const char *)ring + slot * row_bytes,
                              (size_t)n * row_bytes, cudaMemcpyDeviceToHost, st));
        s += n;
        row += n;
    }
    return EXTMCMC_OK;
}

int32_t extmcmc_history_fetch_begin(extmcmc_t h, int64_t seq_lo, int64_t seq_hi) {
    if (!h) return EXTMCMC_EINVAL;
    if (h->fetch_active) return fail(h, EXTMCMC_EINVAL, "a history fetch is already outstanding");
    if (seq_lo < 0 || seq_hi < seq_lo || seq_hi > h->seq_next) return fail(h, EXTMCMC_EINVAL, "bad history range");
    if (seq_lo < h->seq_next - h->d.H) return fail(h, EXTMCMC_ESTALE, "history rows already overwritten");
    CK(h, cudaSetDevice(h->cfg.device));
    const DevState &d = h->d;
    const size_t n = (size_t)(seq_hi - seq_lo), C = (size_t)d.C, rp = (size_t)d.p * C * 8;
    const size_t need = n * (2 * rp + 2 * C * 8 + C);
    if (need > h->stage_cap) {
        CK(h, cudaStreamSynchronize(h->copy_stream));
        if (h->stage) cudaFreeHost(h->stage);
        h->stage = nullptr; h->stage_cap = 0;
        CK(h, cudaMallocHost(&h->stage, need));
        h->stage_cap = need;
    }
    CK(h, cudaEventRecord(h->fetch_ready, h->stream));
    CK(h, cudaStreamWaitEvent(h->copy_stream, h->fetch_ready, 0));
    unsigned char *st = h->stage;
    int32_t rc;
    if ((rc = copy_ring_rows(h, st, d.h_theta, rp, seq_lo, seq_hi, h->copy_stream))) return rc;
    if ((rc = copy_ring_rows(h, st + n * rp, d.h_prop, rp, seq_lo, seq_hi, h->copy_stream))) return rc;
    if ((rc = copy_ring_rows(h, st + 2 * n * rp, d.h_ll, C * 8, seq_lo, seq_hi, h->copy_stream))) return rc;
    if ((rc = copy_ring_rows(h, st + 2 * n * rp + n * C * 8, d.h_llp, C * 8, seq_lo, seq_hi, h->copy_stream))) return rc;
    if ((rc = copy_ring_rows(h, st + 2 * n * rp + 2 * n * C * 8, d.h_acc, C, seq_lo, seq_hi, h->copy_stream))) return rc;
    CK(h, cudaEventRecord(h->fetch_done, h->copy_stream));
    h->fetch_lo = seq_lo; h->fetch_hi = seq_hi;
    h->fetch_active = true;
    return EXTMCMC_OK;
}

int32_t extmcmc_history_fetch_end(extmcmc_t h, double *theta, double *theta_prop, double *ll,
                                  double *ll_prop, uint8_t *accepted) {
    if (!h) return EXTMCMC_EINVAL;
    if (!h->fetch_active) return fail(h, EXTMCMC_EINVAL, "no history fetch outstanding");
    CK(h, cudaEventSynchronize(h->fetch_done));
    h->fetch_active = false;
    const DevState &d = h->d;
    const size_t n = (size_t)(h->fetch_hi - h->fetch_lo), C = (size_t)d.C, rp = (size_t)d.p * C * 8;
    const unsigned char *st = h->stage;
    if (theta) std::memcpy(theta, st, n * rp);
    if (theta_prop) std::memcpy(theta_prop, st + n * rp, n * rp);
    if (ll) std::memcpy(ll, st + 2 * n * rp, n * C * 8);
    if (ll_prop) std::memcpy(ll_prop, st + 2 * n * rp + n * C * 8, n * C * 8);
    if (accepted) std::memcpy(accepted, st + 2 * n * rp + 2 * n * C * 8, n * C);
    return EXTMCMC_OK;
}

int32_t extmcmc_get_stats(extmcmc_t h, double *mean, double *cov, double *rolling_ar,
                          int64_t *n_accept, int64_t *n_prop) {
    if (!h) return EXTMCMC_EINVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    const DevState &d = h->d;
    const int64_t C = d.C;
    if (mean) {
        if (d.stats_mode == 2) return fail(h, EXTMCMC_EINVAL, "running moments disabled (stats_mode = 2)");
        CK(h, cudaMemcpy(mean, d.mean, sizeof(double) * d.p * C, cudaMemcpyDeviceToHost));
    }
    if (cov) {
        if (d.stats_mode == 2) return fail(h, EXTMCMC_EINVAL, "running moments disabled (stats_mode = 2)");
        const size_t covn = d.stats_mode == 0 ? (size_t)d.p * d.p : (size_t)d.p;
        CK(h, cudaMemcpy(cov, d.cov, sizeof(double) * covn * C, cudaMemcpyDeviceToHost));
    }
    for (int u = 0; u < h->cfg.n_updates; ++u) {
        if (!h->upd_set[u]) return fail(h, EXTMCMC_EINVAL, "update not set");
        const DevUpdate &t = h->upd_host[u];
        if (rolling_ar) CK(h, cudaMemcpy(rolling_ar + (size_t)u * C, t.ra_val, sizeof(double) * C, cudaMemcpyDeviceToHost));
        if (n_accept) CK(h, cudaMemcpy(n_accept + (size_t)u * C, t.tot_acc, sizeof(int64_t) * C, cudaMemcpyDeviceToHost));
        if (n_prop) CK(h, cudaMemcpy(n_prop + (size_t)u * C, t.tot_prop, sizeof(int64_t) * C, cudaMemcpyDeviceToHost));
    }
    return EXTMCMC_OK;
}

int32_t extmcmc_get_eps(extmcmc_t h, int32_t u, double *eps) {
    if (!h || !eps) return EXTMCMC_EINVAL;
    if (u < 0 || u >= h->cfg.n_updates || !h->upd_set[u]) return fail(h, EXTMCMC_EINVAL, "update not set");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    const DevUpdate &t = h->upd_host[u];
    if (t.kernel == EXTMCMC_KERNEL_RW_UNIFORM)
        CK(h, cudaMemcpy(eps, t.eps, sizeof(double) * t.n_coords * h->d.C, cudaMemcpyDeviceToHost));
    else if (t.kernel == EXTMCMC_KERNEL_MALA)
        CK(h, cudaMemcpy(eps, t.eps, sizeof(double) * h->d.C, cudaMemcpyDeviceToHost));
    else if (t.kernel == EXTMCMC_KERNEL_RW_GAUSS_MIX)
        CK(h, cudaMemcpy(eps, t.sigB, sizeof(double) * t.n_coords * t.n_coords * h->d.C, cudaMemcpyDeviceToHost));
    else
        return fail(h, EXTMCMC_EINVAL, "this transition kernel has no per-chain step-size state");
    return EXTMCMC_OK;
}

int32_t extmcmc_get_adapt_state(extmcmc_t h, int32_t u, double *mean, double *cov) {
    if (!h) return EXTMCMC_EINVAL;
    if (u < 0 || u >= h->cfg.n_updates || !h->upd_set[u]) return fail(h, EXTMCMC_EINVAL, "update not set");
    const DevUpdate &t = h->upd_host[u];
    if (t.adapt_kind != EXTMCMC_ADAPT_HAARIO) return fail(h, EXTMCMC_EINVAL, "update has no Haario adaptation");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->stream));
    if (mean) CK(h, cudaMemcpy(mean, t.hmean, sizeof(double) * t.n_coords * h->d.C, cudaMemcpyDeviceToHost));
    if (cov) CK(h, cudaMemcpy(cov, t.hcov, sizeof(double) * t.n_coords * t.n_coords * h->d.C, cudaMemcpyDeviceToHost));
    return EXTMCMC_OK;
}

int32_t extmcmc_eval_loglik(extmcmc_t h, double *ll_out) {
    if (!h || !ll_out) return EXTMCMC_EINVAL;
    if (!h->obs_dev || !h->state_set) return fail(h, EXTMCMC_EINVAL, "observations and state required");
    CK(h, cudaSetDevice(h->cfg.device));
    int32_t rc;
    if ((rc = ensure_plan(h))) return rc;
    if ((rc = ensure_total_obs(h))) return rc;
    if (law_self_finished(h->cfg.law)) {
        if ((rc = enqueue_sweep(h, h->cfg.instrument != 0, false, h->d.theta, h->scratch_ll, nullptr))) return rc;
    } else {
        launch_prepare_current(h->d, h->stream);
        if ((rc = enqueue_sweep(h, h->cfg.instrument != 0, false, h->d.theta))) return rc;
        if (!obs_sharded(h) && !h->tail) { launch_reduce_partials(h->d, h->stream); h->launches += 1; }
        launch_finalize_loglik(h->d, h->scratch_ll, h->stream);
        h->launches += 2;
    }
    CK(h, cudaGetLastError());
    CK(h, cudaMemcpyAsync(ll_out, h->scratch_ll, sizeof(double) * h->d.C, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return EXTMCMC_OK;
}

int32_t extmcmc_eval_grad(extmcmc_t h, double *ll_out, double *grad_out) {
    if (!h || !grad_out) return EXTMCMC_EINVAL;
    if (!h->obs_dev || !h->state_set) return fail(h, EXTMCMC_EINVAL, "observations and state required");
    if ((h->cfg.law != EXTMCMC_LAW_GSN_IID_1D && h->cfg.law != EXTMCMC_LAW_HIER_NORMAL &&
         h->cfg.law != EXTMCMC_LAW_LOGISTIC && h->cfg.law != EXTMCMC_LAW_USER) ||
        (h->cfg.law == EXTMCMC_LAW_USER && h->ulaw.loaded && !h->ulaw.grad))
        return fail(h, EXTMCMC_EUNSUPPORTED, "this law has no device gradient");
    if (obs_sharded(h) && !h->comm) return fail(h, EXTMCMC_EINVAL, "EXTMCMC_SHARD_OBS needs extmcmc_comm_init first");
    CK(h, cudaSetDevice(h->cfg.device));
    int32_t rc;
    if ((rc = ensure_plan(h))) return rc;
    if ((rc = ensure_total_obs(h))) return rc;
    if (law_self_finished(h->cfg.law)) {
        if ((rc = enqueue_sweep(h, h->cfg.instrument != 0, true, h->d.theta, h->scratch_ll, h->d.grad_cur))) return rc;
    } else {
        launch_prepare_current(h->d, h->stream);
        if ((rc = enqueue_sweep(h, h->cfg.instrument != 0, true, h->d.theta))) return rc;
        launch_grad_finalize(grad_view(h), h->d.theta, h->scratch_ll, h->d.grad_cur, h->stream);
        h->launches += 2;
    }
    h->grad_valid = true;
    CK(h, cudaGetLastError());
    if (ll_out) CK(h, cudaMemcpyAsync(ll_out, h->scratch_ll, sizeof(double) * h->d.C, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaMemcpyAsync(grad_out, h->d.grad_cur, sizeof(double) * h->d.p * h->d.C, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return EXTMCMC_OK;
}

int32_t extmcmc_timer_start(extmcmc_t h) {
    if (!h) return EXTMCMC_EINVAL;
    CK(h, cudaEventRecord(h->t0, h->stream));
    return EXTMCMC_OK;
}

int32_t extmcmc_timer_stop(extmcmc_t h, float *ms_out) {
    if (!h || !ms_out) return EXTMCMC_EINVAL;
    CK(h, cudaEventRecord(h->t1, h->stream));
    CK(h, cudaEventSynchronize(h->t1));
    CK(h, cudaEventElapsedTime(ms_out, h->t0, h->t1));
    return EXTMCMC_OK;
}

int32_t extmcmc_event_record(extmcmc_t h, int32_t idx) {
    if (!h) return EXTMCMC_EINVAL;
    if (idx < 0 || idx >= 8192) return fail(h, EXTMCMC_EINVAL, "event index out of range");
    if ((size_t)idx >= h->ev_pool.size()) h->ev_pool.resize((size_t)idx + 1, nullptr);
    if (!h->ev_pool[idx]) CK(h, cudaEventCreate(&h->ev_pool[idx]));
    CK(h, cudaEventRecord(h->ev_pool[idx], h->stream));
    return EXTMCMC_OK;
}

int32_t extmcmc_event_elapsed(extmcmc_t h, int32_t i0, int32_t i1, float *ms_out) {
    if (!h || !ms_out) return EXTMCMC_EINVAL;
    if (i0 < 0 || i1 < 0 || (size_t)i0 >= h->ev_pool.size() || (size_t)i1 >= h->ev_pool.size() ||
        !h->ev_pool[i0] || !h->ev_pool[i1])
        return fail(h, EXTMCMC_EINVAL, "event not recorded");
    CK(h, cudaEventSynchronize(h->ev_pool[i1]));
    CK(h, cudaEventElapsedTime(ms_out, h->ev_pool[i0], h->ev_pool[i1]));
    return EXTMCMC_OK;
}

int32_t extmcmc_get_sweep_time(extmcmc_t h, float *ms_total, int64_t *n_launches) {
    if (!h) return EXTMCMC_EINVAL;
    CK(h, cudaStreamSynchronize(h->stream));
    int32_t rc = collect_events(h);
    if (rc) return rc;
    if (ms_total) *ms_total = h->sweep_ms;
    if (n_launches) *n_launches = h->sweep_launches;
    h->sweep_ms = 0.f;
    h->sweep_launches = 0;
    return EXTMCMC_OK;
}

int64_t extmcmc_launch_count(extmcmc_t h) { return h ? h->launches : 0; }

int32_t extmcmc_flush_l2(extmcmc_t h) {
    if (!h) return EXTMCMC_EINVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    if (!h->flush_buf) {
        h->flush_n = (int64_t)(320ll << 20) / 8;  // 320 MiB > 126 MB L2
        CK(h, cudaMalloc(&h->flush_buf, (size_t)h->flush_n * 8));
    }
    launch_flush_l2(h->flush_buf, h->flush_n, h->num_sms, h->stream);
    CK(h, cudaGetLastError());
    return EXTMCMC_OK;
}

int32_t extmcmc_measure_fp64_peak(extmcmc_t h, double *tflops_out) {
    if (!h || !tflops_out) return EXTMCMC_EINVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    const int iters = 16000;   // multiple of the unroll factor 8
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        CK(h, cudaEventRecord(h->t0, h->stream));
        launch_fp64_peak(h->scratch_ll, iters, h->num_sms, h->stream);
        CK(h, cudaEventRecord(h->t1, h->stream));
        CK(h, cudaEventSynchronize(h->t1));
        float ms = 0.f;
        CK(h, cudaEventElapsedTime(&ms, h->t0, h->t1));
        const double flops = (double)h->num_sms * 8 * 256 * 16.0 * iters * 2.0;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    *tflops_out = best;
    return EXTMCMC_OK;
}

int32_t extmcmc_measure_dmma_peak(extmcmc_t h, double *tflops_out) {
    if (!h || !tflops_out) return EXTMCMC_EINVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    const int iters = 4000;
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        CK(h, cudaEventRecord(h->t0, h->stream));
        launch_dmma_peak(h->scratch_ll, iters, h->num_sms, h->stream);
        CK(h, cudaEventRecord(h->t1, h->stream));
        CK(h, cudaEventSynchronize(h->t1));
        float ms = 0.f;
        CK(h, cudaEventElapsedTime(&ms, h->t0, h->t1));
        // warps x 8 independent MMAs x 512 flop (8 x 8 x 4 x 2)
        const double flops = (double)h->num_sms * 8 * 8 /*warps per CTA*/ * 8.0 * iters * 512.0;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    *tflops_out = best;
    return EXTMCMC_OK;
}

const char *extmcmc_sweep_variant_name(extmcmc_t h) {
    if (!h) return "";
    if (!h->plan_valid && h->obs_dev) ensure_plan(h);
    if (!h->plan_valid) return "unplanned";
    bool all_set = true;
    for (int u = 0; u < h->cfg.n_updates; ++u) all_set = all_set && h->upd_set[u];
    if (all_set && plan_block_kernels(h) == EXTMCMC_OK) {
        if (h->res_ok) {
            static const char *rn[] = {"", "", "", "", "team_block_R4", "team_block_R5", "team_block_R6", "team_block_R7", "team_block_R8"};
            return rn[h->res_plan.R];
        }
        if (h->obsblk_ok) {
            const int64_t C = h->d.C;
            return C <= 1 ? "obs_block_C1" : C <= 2 ? "obs_block_C2" : C <= 4 ? "obs_block_C4"
                 : C <= 8 ? "obs_block_C8" : C <= 16 ? "obs_block_C16" : "obs_block_C32";
        }
    }
    return h->plan.name;
}

}  // extern "C"
