// capi.cu -- the extern "C" boundary of libcopra_b200.so (include/copra_b200.h).
// Host-side plumbing only: argument validation (the dimension checks copra performs in
// initializeCost / initializeConstraint), packing of parameter arrays into one pinned staging
// buffer + one H2D copy, device workspace management, kernel sequencing, D2H of the results.
// There is no CPU compute path: every numeric result comes from the sm_100a kernels.
#include "../../include/copra_b200.h"
#include "engine.cuh"
#include "launch.h"
#include "gi_solver.cuh"
#include "gi_thin.cuh"
#include "slice.h"

#include <nvtx3/nvToolsExt.h>

#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <vector>

using namespace cb;

namespace {

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
};

struct Sizes {
    int X = 0, nU = 0, nvar = 0, meq = 0, mineq = 0, q = 0;
};

} // namespace

struct copra_b200_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sms = 148;
    size_t smem_optin = 227 * 1024;
    int plan_sms = 148;     // SMs the solver planners size their grids for: sms, or copra_b200_options::sm_limit if smaller
    int small_variant = 0;  // copra_b200_options::small_variant
    std::string err;
    long long launches = 0;
    long long call_launches = 0;
    std::map<std::string, Buf> dev;
    Buf pin_in, pin_out;
    cudaEvent_t ev[8] = {};
    bool ev_valid[8] = {};
    cudaEvent_t h2d_done = nullptr; // guards reuse of the pinned upload staging buffer
    bool h2d_pending = false;
    // TrajectoryBound line selection cache for DEVICE inputs: (lower ptr, upper ptr, rows, full_size) -> lines
    struct TbKey {
        const double* lo; const double* up; int rows, full_size;
        bool operator<(const TbKey& o) const { return std::tie(lo, up, rows, full_size) < std::tie(o.lo, o.up, o.rows, o.full_size); }
    };
    std::map<TbKey, std::pair<std::vector<int>, std::vector<int>>> tb_cache;
    std::vector<double> sel_host; // last uploaded selector matrices / line lists
    std::vector<int> lines_host;
    // state of the last build
    bool built = false;
    std::vector<int> shape;    // shape_key() of the last build: what copra_b200_lmpc_retarget must find unchanged
    bool factor_valid = false; // the thin solver's R^-1 of the last build is resident (re-solves skip the factorisation)
    bool rows_filled = false;  // Aeq / Aineq of the last build are materialised (the structured solver never reads them)
    bool use_thin = false;     // the last build is solved by the thin kernel (gi_thin.cuh)
    bool gs_j_valid = false;   // the small solver's per-instance factors of the resident build are cached (re-solves load them)
    bool warm_start = false;   // copra_b200_set_warm_start: re-solves seed the active set of the previous solve
    bool warm_valid = false;   // `warm_iact` holds the active sets of the last solve of the resident build
    bool solved = false;       // res_x / res_status / res_nact / res_iact hold the last solve of the resident build (lmpc_vjp)
    bool vjp_factor_valid = false; // vjp_Jt holds R^-1 of the resident build's Hessian(s) (builds the thin solver did not factor)
    // the last raw QP batch (copra_b200_qp_vjp): its shape and input arrays (the caller's device arrays, or the qp_params
    // staging buffer), its solution in res_x / res_status / res_nact / res_iact; any LMPC call clears qp_solved
    bool qp_solved = false;
    GiBatch qp{};
    // per-instance vector lengths of the resident build (doubles): every cost's p, every constraint's f / lower / upper;
    // the constraint and the side (0 f, 1 lower, 2 upper) of every family; the control-bound constraint (-1 = none)
    std::vector<int> cost_len, cstr_len, fam_cstr, fam_which;
    int bound_cstr = -1;
    bool in_resolve = false;
    bool lmpc_solve_active = false; // run_gi is called from do_solve (a resident LMPC build), not from the raw-QP entry
    bool gt_shared = false;    // ... with a batch-invariant system and Hessian (one factor, the Dpsi / Hpsi tables)
    bool gt_pform = false;     // ... in its shared-factor form (P = Jt Q1 kept, no factor mat-vec per pass)
    const char* solver = "";   // K5+K6 kernel(s) of the last solve
    bool nvtx_open = false;    // an NVTX stage range is open on the calling thread
    GtBatch gt{};
    GtPlan gtplan{};
    BuildParams bp{};
    Sizes sz;
    double vsmall = 0;
    double fp64_peaks[2] = { 0.0, 0.0 }; // measured DFMA / DMMA TFLOP/s (lazy)
};

namespace {

int fail(copra_b200_handle* h, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

#define LAUNCHED(expr)                                                                                              \
    do {                                                                                                            \
        int n_ = (expr);                                                                                            \
        if (n_ < 0) return fail(h, COPRA_B200_E_CUDA, "%s: %s", #expr, cudaGetErrorString(cudaError_t(-n_)));        \
        h->launches += n_;                                                                                          \
        h->call_launches += n_;                                                                                     \
    } while (0)

int dev_reserve(copra_b200_handle* h, const char* name, size_t bytes, void** out)
{
    Buf& b = h->dev[name];
    if (bytes > b.cap) {
        if (b.p) CU(cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
        size_t cap = bytes + bytes / 8 + 256;
        CU(cudaMalloc(&b.p, cap));
        b.cap = cap;
    }
    *out = b.p;
    return 0;
}

int pin_reserve(copra_b200_handle* h, Buf& b, size_t bytes)
{
    if (bytes > b.cap) {
        if (b.p) CU(cudaFreeHost(b.p));
        b.p = nullptr;
        b.cap = 0;
        size_t cap = bytes + bytes / 8 + 256;
        CU(cudaMallocHost(&b.p, cap));
        b.cap = cap;
    }
    return 0;
}

// Stage boundaries: CUDA event k on the stream (copra_b200_last_timing) + an NVTX range per stage for Nsight timelines
// (SURVEY.md 5: the reference's only tracing is the two wall-clock timers of src/LMPC.cpp:82-99).
int record(copra_b200_handle* h, int k)
{
    static const char* const kStage[6] = { "copra_b200: H2D parameters", "copra_b200: K1 condense", "copra_b200: K2-K4 assemble",
        "copra_b200: K5+K6 solve", "copra_b200: K7 rollout", "copra_b200: D2H results" };
    if (h->nvtx_open) { nvtxRangePop(); h->nvtx_open = false; }
    if (k >= 0 && k < 6) { nvtxRangePushA(kStage[k]); h->nvtx_open = true; }
    if (!h->ev[k]) CU(cudaEventCreate(&h->ev[k]));
    CU(cudaEventRecord(h->ev[k], h->stream));
    h->ev_valid[k] = true;
    return 0;
}

// ---- staged upload of (ptr, stride) arrays ----------------------------------------------------
struct Upload {
    struct Item {
        copra_b200_array src;
        size_t size;   // doubles per instance
        DArr* dst;
        size_t offset; // doubles into the packed buffer
        bool shared;
    };
    std::vector<Item> items;
    size_t total = 0;
    void add(copra_b200_array a, size_t size, DArr* dst)
    {
        if (!a.ptr || size == 0) { dst->p = nullptr; dst->s = 0; return; }
        Item it{ a, size, dst, 0, a.stride == 0 };
        items.push_back(it);
    }
};

int run_upload(copra_b200_handle* h, Upload& U, int batch, int memory, const char* bufname)
{
    if (memory == COPRA_B200_DEVICE) {
        for (auto& it : U.items) { it.dst->p = it.src.ptr; it.dst->s = it.src.stride; }
        return 0;
    }
    size_t total = 0;
    for (auto& it : U.items) {
        it.offset = total;
        total += it.shared ? it.size : it.size * size_t(batch);
        total = (total + 1) & ~size_t(1); // keep 16-byte alignment
        if (!it.shared && it.src.stride < (long long)it.size)
            return fail(h, COPRA_B200_E_ARG, "array stride %lld smaller than its per-instance size %zu", it.src.stride, it.size);
    }
    if (total == 0) return 0;
    int rc = pin_reserve(h, h->pin_in, total * sizeof(double));
    if (rc) return rc;
    void* dptr = nullptr;
    rc = dev_reserve(h, bufname, total * sizeof(double), &dptr);
    if (rc) return rc;
    if (h->h2d_pending) { CU(cudaEventSynchronize(h->h2d_done)); h->h2d_pending = false; }
    double* stage = static_cast<double*>(h->pin_in.p);
    for (auto& it : U.items) {
        double* d = stage + it.offset;
        if (it.shared) std::memcpy(d, it.src.ptr, it.size * sizeof(double));
        else if (it.src.stride == (long long)it.size) std::memcpy(d, it.src.ptr, it.size * size_t(batch) * sizeof(double));
        else
            for (int b = 0; b < batch; ++b) std::memcpy(d + size_t(b) * it.size, it.src.ptr + (long long)b * it.src.stride, it.size * sizeof(double));
        it.dst->p = static_cast<double*>(dptr) + it.offset;
        it.dst->s = it.shared ? 0 : (long long)it.size;
    }
    CU(cudaMemcpyAsync(dptr, stage, total * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if (!h->h2d_done) CU(cudaEventCreateWithFlags(&h->h2d_done, cudaEventDisableTiming));
    CU(cudaEventRecord(h->h2d_done, h->stream));
    h->h2d_pending = true;
    return 0;
}

// copy a device result to the caller (device->device or device->host through pinned staging)
struct Download {
    struct Item {
        const void* src;
        void* dst;
        size_t bytes;
        size_t offset;
    };
    std::vector<Item> items;
    void add(const void* src, void* dst, size_t bytes)
    {
        if (dst && bytes) items.push_back(Item{ src, dst, bytes, 0 });
    }
};

int run_download(copra_b200_handle* h, Download& D, int memory)
{
    if (D.items.empty()) return 0;
    if (memory == COPRA_B200_DEVICE) {
        for (auto& it : D.items)
            if (it.src != it.dst) CU(cudaMemcpyAsync(it.dst, it.src, it.bytes, cudaMemcpyDeviceToDevice, h->stream));
        return 0;
    }
    // page-locked destinations (cudaMallocHost / torch pinned tensors) are written by DMA directly; pageable ones go
    // through the handle's pinned staging buffer
    size_t total = 0;
    std::vector<char> direct(D.items.size(), 0);
    for (size_t k = 0; k < D.items.size(); ++k) {
        auto& it = D.items[k];
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, it.dst) == cudaSuccess && attr.type == cudaMemoryTypeHost) direct[k] = 1;
        else { cudaGetLastError(); it.offset = total; total += (it.bytes + 15) & ~size_t(15); }
    }
    int rc = pin_reserve(h, h->pin_out, total);
    if (rc) return rc;
    char* stage = static_cast<char*>(h->pin_out.p);
    for (size_t k = 0; k < D.items.size(); ++k) {
        auto& it = D.items[k];
        CU(cudaMemcpyAsync(direct[k] ? it.dst : static_cast<void*>(stage + it.offset), it.src, it.bytes, cudaMemcpyDeviceToHost, h->stream));
    }
    CU(cudaStreamSynchronize(h->stream));
    for (size_t k = 0; k < D.items.size(); ++k)
        if (!direct[k]) std::memcpy(D.items[k].dst, stage + D.items[k].offset, D.items[k].bytes);
    return 0;
}

// ---- problem description -> families ----------------------------------------------------------
struct Plan {
    Sizes sz;
    // vsteps: steps held by the vector (p, f, lower / upper) of a per-step entry, 1 otherwise; pstep / fstep: the
    // family's stride between steps (0 = the same vector at every step)
    struct CostMeta { int kind, rows, i0, i1, hasM, hasN, dense, vsteps, pstep; };
    struct FamMeta { int cstr, rows, i0, i1, hasE, hasG, is_eq, row_off, which, dense, gather, fstep; std::vector<int> lines; };
    int cb_full = 0;
    std::vector<CostMeta> costs;
    std::vector<FamMeta> fams;
    std::vector<int> cvsteps; // per constraint
    int bound_cstr = -1;
};

int fetch_host(copra_b200_handle* h, const copra_b200_array& a, int count, int memory, std::vector<double>& out)
{
    out.resize(count);
    if (memory == COPRA_B200_HOST) std::memcpy(out.data(), a.ptr, sizeof(double) * count);
    else {
        CU(cudaMemcpyAsync(out.data(), a.ptr, sizeof(double) * count, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

// vectors_only: the problem only supplies new vectors for a resident build (copra_b200_lmpc_retarget), so the matrices
// may be absent
int make_plan(copra_b200_handle* h, const copra_b200_problem* p, Plan& pl, bool vectors_only = false)
{
    if (!p) return fail(h, COPRA_B200_E_ARG, "null problem");
    if (p->nx <= 0 || p->nu <= 0 || p->batch <= 0) return fail(h, COPRA_B200_E_ARG, "nx, nu and batch must be positive");
    if (p->N <= 0) return fail(h, COPRA_B200_E_ARG, "The number of step sould be a positive number!"); // PreviewSystem.cpp:31-33
    if (!p->x0.ptr || (!vectors_only && (!p->A.ptr || !p->B.ptr || !p->d.ptr))) return fail(h, COPRA_B200_E_ARG, "A, B, d and x0 are required");
    if (p->ncost < 0 || p->ncost > kMaxCost) return fail(h, COPRA_B200_E_ARG, "at most %d cost functions", kMaxCost);
    if (p->memory != COPRA_B200_HOST && p->memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    const int nx = p->nx, nu = p->nu, N = p->N;
    pl.sz.X = nx * (N + 1);
    pl.sz.nU = nu * N;
    pl.sz.nvar = p->initial_state ? nx + pl.sz.nU : pl.sz.nU;
    for (int i = 0; i < p->ncost; ++i) {
        const copra_b200_cost& c = p->costs[i];
        if (c.rows <= 0 || !c.p.ptr) return fail(h, COPRA_B200_E_ARG, "cost %d: rows must be positive and p given", i);
        if (c.full_size < 0 || c.full_size > COPRA_B200_PER_STEP) return fail(h, COPRA_B200_E_ARG, "cost %d: full_size must be 0, 1 or COPRA_B200_PER_STEP", i);
        Plan::CostMeta m{ c.kind, c.rows, 0, 0, 0, 0, c.full_size == 1 ? 1 : 0, 1, 0 };
        switch (c.kind) {
        case COPRA_B200_COST_TRAJECTORY: m.i0 = 0; m.i1 = N + 1; m.hasM = 1; break;
        case COPRA_B200_COST_TARGET: m.i0 = N; m.i1 = N + 1; m.hasM = 1; break;
        case COPRA_B200_COST_CONTROL: m.i0 = 0; m.i1 = N; m.hasN = 1; break;
        case COPRA_B200_COST_MIXED: m.i0 = 0; m.i1 = N; m.hasM = 1; m.hasN = 1; break;
        default: return fail(h, COPRA_B200_E_ARG, "cost %d: unknown kind %d", i, c.kind);
        }
        if (!vectors_only) {
            if (m.hasM && !c.M.ptr) return fail(h, COPRA_B200_E_ARG, "cost %d: M is required", i);
            if (m.hasN && !c.N.ptr) return fail(h, COPRA_B200_E_ARG, "cost %d: N is required", i);
            if (!c.w.ptr) return fail(h, COPRA_B200_E_ARG, "cost %d: weights are required (copra default: ones)", i);
        }
        if (c.full_size == COPRA_B200_PER_STEP) {
            if (c.kind == COPRA_B200_COST_TARGET) return fail(h, COPRA_B200_E_ARG, "cost %d: a TargetCost has one step: it takes no per-step p", i);
            m.vsteps = m.i1 - m.i0;
            m.pstep = c.rows;
        }
        if (m.dense) {
            if (c.kind == COPRA_B200_COST_TARGET) return fail(h, COPRA_B200_E_ARG, "cost %d: TargetCost takes a step-size M (xDim columns) only", i);
            m.i0 = 0; m.i1 = 1; // one stacked block
        }
        pl.costs.push_back(m);
    }
    int eq_off = 0, in_off = 0;
    for (int i = 0; i < p->ncstr; ++i) {
        const copra_b200_constraint& c = p->cstrs[i];
        if (c.rows <= 0) return fail(h, COPRA_B200_E_ARG, "constraint %d: rows must be positive", i);
        if (c.full_size < 0 || c.full_size > COPRA_B200_PER_STEP)
            return fail(h, COPRA_B200_E_ARG, "constraint %d: full_size must be 0, 1 or COPRA_B200_PER_STEP", i);
        const bool full = c.full_size == 1, per_step = c.full_size == COPRA_B200_PER_STEP;
        // steps of the horizon the constraint applies to: its vector holds that many copies when given per step
        const int steps = (c.kind == COPRA_B200_CSTR_TRAJECTORY || c.kind == COPRA_B200_CSTR_TRAJECTORY_BOUND) ? N + 1 : N;
        pl.cvsteps.push_back(per_step ? steps : 1);
        auto push = [&](int i0, int i1, int hasE, int hasG, bool iseq, int which, std::vector<int> lines) {
            Plan::FamMeta f;
            f.cstr = i; f.rows = lines.empty() ? c.rows : int(lines.size());
            f.dense = (full && which == 0) ? 1 : 0;
            f.gather = (full && which != 0) ? 1 : 0;
            f.fstep = per_step ? c.rows : 0; // a trajectory bound's rows are nx: its vectors hold every line of a step
            if (full) { i0 = 0; i1 = 1; }
            f.i0 = i0; f.i1 = i1; f.hasE = hasE; f.hasG = hasG; f.is_eq = iseq ? 1 : 0; f.which = which;
            f.lines = std::move(lines);
            int& off = iseq ? eq_off : in_off;
            f.row_off = off;
            off += f.rows * (i1 - i0);
            pl.fams.push_back(f);
        };
        switch (c.kind) {
        case COPRA_B200_CSTR_TRAJECTORY:
            if ((!vectors_only && !c.E.ptr) || !c.f.ptr) return fail(h, COPRA_B200_E_ARG, "constraint %d: E and f are required", i);
            push(0, N + 1, 1, 0, !c.is_ineq, 0, {});
            break;
        case COPRA_B200_CSTR_CONTROL:
            if ((!vectors_only && !c.G.ptr) || !c.f.ptr) return fail(h, COPRA_B200_E_ARG, "constraint %d: G and f are required", i);
            push(0, N, 0, 1, !c.is_ineq, 0, {});
            break;
        case COPRA_B200_CSTR_MIXED:
            if ((!vectors_only && (!c.E.ptr || !c.G.ptr)) || !c.f.ptr) return fail(h, COPRA_B200_E_ARG, "constraint %d: E, G and f are required", i);
            push(0, N, 1, 1, !c.is_ineq, 0, {});
            break;
        case COPRA_B200_CSTR_TRAJECTORY_BOUND: {
            if (!c.lower.ptr || !c.upper.ptr) return fail(h, COPRA_B200_E_ARG, "constraint %d: lower and upper are required", i);
            const int brows = full ? pl.sz.X : nx, count = brows * pl.cvsteps.back();
            if (c.rows != brows) return fail(h, COPRA_B200_E_ARG, "constraint %d: trajectory bounds must have xDim (or fullXDim) rows", i);
            // line selection (include/constraints.h:247-254) is part of the problem SHAPE: it is taken
            // from instance 0 and verified to be the same at every step of a per-step entry and, for host inputs, for every
            // instance.
            std::vector<int> ll, ul;
            copra_b200_handle::TbKey key{ c.lower.ptr, c.upper.ptr, brows, c.full_size };
            auto hit = h->tb_cache.find(key);
            // DEVICE inputs: the +-inf pattern is read back from instance 0 on EVERY build (one small D2H + sync) unless the
            // caller vouches with COPRA_B200_FLAG_STABLE_BOUND_PATTERN that it has not changed since the last build that
            // used these pointers (a rewritten or re-allocated bound tensor would otherwise reuse stale line lists)
            const bool may_cache = p->memory == COPRA_B200_DEVICE && (p->flags & COPRA_B200_FLAG_STABLE_BOUND_PATTERN);
            if (may_cache && hit != h->tb_cache.end()) {
                ll = hit->second.first;
                ul = hit->second.second;
            } else {
                std::vector<double> lo, up;
                int rc = fetch_host(h, c.lower, count, p->memory, lo);
                if (rc) return rc;
                rc = fetch_host(h, c.upper, count, p->memory, up);
                if (rc) return rc;
                for (int l = 0; l < brows; ++l) if (lo[l] != -INFINITY) ll.push_back(l);
                for (int l = 0; l < brows; ++l) if (up[l] != INFINITY) ul.push_back(l);
                const int nb = p->memory == COPRA_B200_HOST ? p->batch : 1;
                for (int b = 0; b < nb; ++b)
                    for (int l = 0; l < count; ++l) {
                        const double a = b ? c.lower.ptr[(long long)b * c.lower.stride + l] : lo[l];
                        const double u = b ? c.upper.ptr[(long long)b * c.upper.stride + l] : up[l];
                        if ((a != -INFINITY) != (lo[l % brows] != -INFINITY) || (u != INFINITY) != (up[l % brows] != INFINITY))
                            return fail(h, COPRA_B200_E_ARG, "constraint %d: the set of infinite trajectory bounds must be the same at every step and for every instance", i);
                    }
                if (may_cache) {
                    if (h->tb_cache.size() > 64) h->tb_cache.clear();
                    h->tb_cache[key] = std::make_pair(ll, ul);
                }
            }
            if (!ll.empty()) push(0, N + 1, 1, 0, false, 1, ll);
            if (!ul.empty()) push(0, N + 1, 1, 0, false, 2, ul);
        } break;
        case COPRA_B200_CSTR_CONTROL_BOUND:
            if (!c.lower.ptr || !c.upper.ptr) return fail(h, COPRA_B200_E_ARG, "constraint %d: lower and upper are required", i);
            if (c.rows != (full ? pl.sz.nU : nu)) return fail(h, COPRA_B200_E_ARG, "constraint %d: control bounds must have uDim (or fullUDim) rows", i);
            pl.cb_full = (full || per_step) ? 1 : 0; // a per-step lower / upper holds the nU entries of a full-size one
            if (pl.bound_cstr >= 0) return fail(h, COPRA_B200_E_UNSUPPORTED, "only one ControlBoundConstraint per controller (reference quirk Q8)");
            pl.bound_cstr = i;
            break;
        default: return fail(h, COPRA_B200_E_ARG, "constraint %d: unknown kind %d", i, c.kind);
        }
    }
    if (int(pl.fams.size()) > kMaxFam) return fail(h, COPRA_B200_E_ARG, "too many constraint families");
    pl.sz.meq = eq_off;
    pl.sz.mineq = in_off;
    pl.sz.q = eq_off + in_off + 2 * pl.sz.nvar;
    return 0;
}

// Everything a build fixes besides the matrices: dimensions, every entry's kind, rows, form and inequality sense, and the
// trajectory-bound line selections.  A retarget must find it unchanged.
std::vector<int> shape_key(const copra_b200_problem* p, const Plan& pl)
{
    std::vector<int> k{ p->nx, p->nu, p->N, p->batch, p->initial_state ? 1 : 0, p->ncost, p->ncstr };
    for (int i = 0; i < p->ncost; ++i) k.insert(k.end(), { p->costs[i].kind, p->costs[i].rows, p->costs[i].full_size });
    for (int i = 0; i < p->ncstr; ++i) {
        const copra_b200_constraint& c = p->cstrs[i];
        const bool rowcs = c.kind != COPRA_B200_CSTR_TRAJECTORY_BOUND && c.kind != COPRA_B200_CSTR_CONTROL_BOUND;
        k.insert(k.end(), { c.kind, c.rows, c.full_size, rowcs ? (c.is_ineq ? 1 : 0) : 0 });
    }
    for (const auto& f : pl.fams) {
        k.push_back(int(f.lines.size()));
        k.insert(k.end(), f.lines.begin(), f.lines.end());
    }
    return k;
}

// The per-instance vectors of a problem: x0, every cost's p, every constraint's f / lower / upper (rows x steps doubles
// per instance for a per-step entry).  A build uploads them with its matrices, a retarget alone.
struct BoundArrs { std::vector<DArr> lower, upper; };

void add_vectors(Upload& U, const copra_b200_problem* p, const Plan& pl, BuildParams& P, BoundArrs& ba)
{
    U.add(p->x0, P.nx, &P.x0);
    for (int i = 0; i < P.ncost; ++i) {
        const copra_b200_cost& c = p->costs[i];
        U.add(c.p, size_t(c.rows) * pl.costs[i].vsteps, &P.cost[i].p);
    }
    // trajectory-bound families share the uploaded lower / upper vectors of their constraint
    ba.lower.assign(p->ncstr, DArr{ nullptr, 0 });
    ba.upper.assign(p->ncstr, DArr{ nullptr, 0 });
    for (int i = 0; i < p->ncstr; ++i) {
        const copra_b200_constraint& c = p->cstrs[i];
        if (c.kind == COPRA_B200_CSTR_TRAJECTORY_BOUND || c.kind == COPRA_B200_CSTR_CONTROL_BOUND) {
            U.add(c.lower, size_t(c.rows) * pl.cvsteps[i], &ba.lower[i]);
            U.add(c.upper, size_t(c.rows) * pl.cvsteps[i], &ba.upper[i]);
        }
    }
    for (int k = 0; k < P.nfam; ++k) {
        const auto& f = pl.fams[k];
        const copra_b200_constraint& c = p->cstrs[f.cstr];
        if (f.which == 0) U.add(c.f, size_t(c.rows) * pl.cvsteps[f.cstr], &P.fam[k].f);
    }
}

// after run_upload: point the bound families and the control bounds at the uploaded lower / upper
void bind_bounds(const Plan& pl, BuildParams& P, const BoundArrs& ba)
{
    for (int k = 0; k < P.nfam; ++k) {
        const auto& f = pl.fams[k];
        if (f.which != 0) P.fam[k].f = f.which == 1 ? ba.lower[f.cstr] : ba.upper[f.cstr];
    }
    if (pl.bound_cstr >= 0) {
        P.cb_lower = ba.lower[pl.bound_cstr];
        P.cb_upper = ba.upper[pl.bound_cstr];
        P.cb_full = pl.cb_full;
    }
}

template <class T> int ws(copra_b200_handle* h, const char* name, size_t count, T** out)
{
    void* p = nullptr;
    int rc = dev_reserve(h, name, std::max<size_t>(count, 1) * sizeof(T), &p);
    *out = static_cast<T*>(p);
    return rc;
}

// Launch K5+K6 for a prepared batch: picks the small / single-CTA / cluster variant and provides the
// workspace each needs.  Returns 0 or a negative C-ABI code; counts the kernels it launched.
int run_gi(copra_b200_handle* h, GiBatch& G)
{
    int rc;
    GiPlan plan = gi_plan(G.n, G.meq, G.m, G.batch, h->plan_sms, h->smem_optin, h->small_variant);
    int* counter = nullptr;
    if ((rc = ws(h, "counter", 2, &counter))) return rc;
    CU(cudaMemsetAsync(counter, 0, 2 * sizeof(int), h->stream));
    G.counter = counter;
    G.vsmall = h->vsmall;
    G.max_iter = 50 * (G.meq + G.m + 2 * G.n) + 100;
    G.j_smem = plan.j_smem; G.s_smem = plan.s_smem; G.a_smem = plan.a_smem;
    G.ws = nullptr; G.ws_stride = plan.ws_stride;
    h->solver = plan.small ? "gi_small_kernel" : "gi_batch_kernel";
    G.jcache = nullptr; G.jflag = nullptr; G.jmode = 0;
    if (plan.small && h->lmpc_solve_active) {
        // re-solves of a resident LMPC build: the first one stores every instance's factor, the following ones load it
        // (<= 2 GB of cache; a plain build + solve pays nothing)
        const int n2e = (G.n + 1) & ~1;
        const size_t per = size_t((n2e % 4 == 2) ? n2e : n2e + 2) * n2e; // ld_vec2(n) * even(n), the kernel's layout of J
        if (per * G.batch * sizeof(double) <= (size_t(2) << 30)) {
            if ((rc = ws(h, "gs_jcache", per * G.batch, &G.jcache))) return rc;
            if ((rc = ws(h, "gs_jflag", size_t(G.batch), &G.jflag))) return rc;
            // (the workspace is reserved by the first solve of the build so that no re-solve allocates)
            if (h->in_resolve) { G.jmode = h->gs_j_valid ? 2 : 1; h->gs_j_valid = true; }
            else { G.jcache = nullptr; G.jflag = nullptr; }
        }
    }
    if (plan.cluster > 0) {
        int nclusters = gi_cluster_max_clusters(plan);
        if (nclusters > 0) {
            h->solver = "gi_cluster_kernel";
            nclusters = std::min(nclusters, G.batch);
            const size_t n = G.n;
            double* Sws = nullptr;
            if ((rc = ws(h, "gi_S", size_t(nclusters) * odd_ld(G.n) * n, &Sws))) return rc;
            cudaError_t e = gi_cluster_launch(G, plan, Sws, nclusters, h->stream);
            if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gi_cluster_launch: %s", cudaGetErrorString(e));
            h->launches += 1; h->call_launches += 1;
            return 0;
        }
        // clusters of this size cannot be scheduled on this device: fall back to the single-CTA variant
        plan.cluster = 0;
        plan.threads = 512; plan.j_smem = plan.s_smem = plan.a_smem = 0;
        plan.smem_bytes = gi_layout(G.n, G.meq, G.m, 512, 0, 0, 0).bytes;
        plan.ws_stride = 2LL * odd_ld(G.n) * G.n;
        plan.grid = std::max(1, std::min(G.batch, h->plan_sms));
        G.j_smem = G.s_smem = G.a_smem = 0;
        G.ws_stride = plan.ws_stride;
    }
    if (plan.ws_stride > 0 && (rc = ws(h, "gi_ws", size_t(plan.grid) * plan.ws_stride, &G.ws))) return rc;
    cudaError_t e = gi_launch(G, plan, h->stream);
    if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gi_launch: %s", cudaGetErrorString(e));
    h->launches += 1; h->call_launches += 1;
    return 0;
}

// Decide whether the build in h->bp goes to the thin solver (gi_thin.cuh): LMPC mode, more variables than the small
// kernel takes, and every general row a step-size (block-Toeplitz) row whose tables fit shared memory.
bool plan_thin(copra_b200_handle* h)
{
    const BuildParams& P = h->bp;
    h->use_thin = false;
    if (P.initial_state) return false;
    const int sms = h->plan_sms;
    const GiPlan legacy = gi_plan(P.nvar, P.meq, P.mineq, P.batch, sms, h->smem_optin, h->small_variant);
    if (legacy.small) return false;
    // a handful of instances: the cluster kernel spreads ONE instance over several SMs (latency); the thin kernel is the
    // throughput design (one SM per instance) and wins as soon as the clusters would not cover the batch in one wave
    if (legacy.cluster > 0 && P.batch * legacy.cluster * 2 <= sms) return false;
    GtBatch& T = h->gt;
    std::memset(&T, 0, sizeof T);
    T.n = P.nvar; T.meq = P.meq; T.m = P.mineq; T.batch = P.batch;
    T.structured = 1; T.nu = P.nu; T.N = P.N; T.nfam = P.nfam;
    int tab = 0;
    for (int k = 0; k < P.nfam; ++k) {
        const CstrFam& F = P.fam[k];
        if (F.dense || F.gather) return false;
        GtFam& f = T.fam[k];
        f.rows = F.rows; f.i0 = F.i0; f.i1 = F.i1; f.is_eq = F.is_eq; f.row_off = F.row_off;
        f.tab = tab;
        tab += F.rows * P.nu * ((P.N + 1) | 1);
    }
    T.tab_doubles = tab;
    T.ldk = (P.N + 1) | 1;
    T.ld = gt_even(T.n);
    T.reorth = 1e-2;
    // state-space evaluation of the general rows (chunks of 16 steps) when its tables fit next to everything else
    T.nx = P.nx; T.X = P.X;
    T.ssL = 16;
    T.ssC = (P.N + T.ssL - 1) / T.ssL;
    int eg = 0;
    for (int k = 0; k < P.nfam; ++k) eg += P.fam[k].rows * ((P.fam[k].hasE ? P.nx : 0) + (P.fam[k].hasG ? P.nu : 0));
    T.ss_doubles = gt_ss_layout(P.nx, P.nu, P.N, T.ssL, T.ssC, eg).total;
    T.ss = P.meq + P.mineq > 0 ? 1 : 0;
    if (!T.ss) T.ss_doubles = 0;
    // batch-invariant system AND Hessian: Dpsi / Hpsi tables and the P form of the pass (see GtBatch)
    const bool shared = P.sQ == 0 && P.A.s == 0 && P.B.s == 0;
    GtShape shape{ T.n, T.meq, T.m, tab, T.ldk, T.ld, T.ss_doubles, shared ? 1 : 0 };
    h->gtplan = gt_plan(shape, T.batch, sms, h->smem_optin);
    if (shape.pform && T.n > h->gtplan.threads) { shape.pform = 0; h->gtplan = gt_plan(shape, T.batch, sms, h->smem_optin); }
    if (T.ss && !h->gtplan.ok) { // does not fit: convolution form
        T.ss = 0; T.ss_doubles = 0; shape.ss_doubles = 0;
        h->gtplan = gt_plan(shape, T.batch, sms, h->smem_optin);
    }
    // Per-instance factors and big streams (n >= 512) in a batch of only a few waves: the step is the latency of its heaviest
    // instance, which is bound by what ONE SM can stream -- give every instance a thread-block cluster instead.
    // 16 CTAs per instance (a non-portable cluster size: one cluster per GPC) when the device schedules them, else 8:
    // C5's heaviest instance takes 0.39 s on 16 CTAs, 0.53 s on 8, 2.3 s on one
    if (P.sQ != 0 && T.n >= 512 && P.batch <= 16 * sms) {
        for (int csize = 16; csize > 1 && h->gtplan.ok; csize >>= 1) {
            GtShape cs = shape;
            cs.cluster = csize; cs.pform = 0; cs.ss_doubles = 0;
            const GtPlan cp = gt_plan(cs, T.batch, sms, h->smem_optin);
            if (cp.ok) { h->gtplan = cp; shape = cs; T.ss = 0; T.ss_doubles = 0; break; }
        }
    }
    if (!h->gtplan.ok) return false;
    h->gt_shared = shared;
    h->gt_pform = shape.pform != 0;
    T.lay = gt_layout(T.n, T.meq, T.m, T.tab_doubles, h->gtplan.threads, h->gtplan.q1s, T.ss_doubles);
    T.ssl = gt_ss_layout(P.nx, P.nu, P.N, T.ssL, T.ssC, eg);
    T.q1s = h->gtplan.q1s;
    h->use_thin = true;
    return true;
}

int run_gt(copra_b200_handle* h, double* x, int* status, int* iters, int* nact, int* iact)
{
    const BuildParams& P = h->bp;
    GtBatch& T = h->gt;
    const GtPlan& plan = h->gtplan;
    const size_t n = P.nvar, ldj = size_t(T.ld), count = P.sQ ? size_t(P.batch) : 1;
    int rc;
    double *Jt = nullptr, *JtT = nullptr, *wsp = nullptr;
    int *pd = nullptr, *counter = nullptr;
    if ((rc = ws(h, "gt_Jt", count * ldj * n, &Jt))) return rc;
    if ((rc = ws(h, "gt_JtT", count * ldj * n, &JtT))) return rc;
    if ((rc = ws(h, "gt_pd", count, &pd))) return rc;
    if ((rc = ws(h, "gt_ws", size_t(plan.grid) * plan.ws_stride, &wsp))) return rc;
    if ((rc = ws(h, "counter", 2, &counter))) return rc;
    // batch-invariant system and Hessian: Dpsi = Jt' Psi' once per build (one Toeplitz fill + one DMMA GEMM)
    const bool use_dpsi = h->gt_shared, pform = h->gt_pform;
    double *psit = nullptr, *dpsi = nullptr, *hpsi = nullptr, *hm = nullptr;
    if (use_dpsi) {
        if ((rc = ws(h, "gt_psit", n * size_t(P.X), &psit))) return rc;
        if ((rc = ws(h, "gt_dpsi", ldj * size_t(P.X), &dpsi))) return rc;
    }
    if (pform) {
        if ((rc = ws(h, "gt_hpsi", ldj * size_t(P.X), &hpsi))) return rc;
        if ((rc = ws(h, "gt_hm", ldj * n, &hm))) return rc;
    }
    if (!h->factor_valid) {
        cudaError_t e = gt_factor_launch(DArr{ P.Q, P.sQ }, P.nvar, T.ld, int(count), Jt, JtT, pd, h->plan_sms, h->stream);
        if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gt_factor_launch: %s", cudaGetErrorString(e));
        h->launches += 1; h->call_launches += 1;
        if (use_dpsi) {
            e = gt_psit_fill_launch(P.Gs, psit, P.nx, P.nu, P.N, h->stream);
            if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gt_psit_fill_launch: %s", cudaGetErrorString(e));
            h->launches += 1; h->call_launches += 1;
            LAUNCHED(dgemm_dmma_launch(1, P.nvar, P.X, P.nvar, 1.0, Jt, T.ld, 0, psit, P.nvar, 0, 0.0, dpsi, T.ld, 0, 1, h->stream));
        }
        if (pform) { // Hpsi = Jt Dpsi (= Q^-1 Psi'), H = Jt Jt' (= Q^-1)
            if (T.ld != P.nvar) {
                CU(cudaMemsetAsync(hpsi, 0, ldj * size_t(P.X) * sizeof(double), h->stream));
                CU(cudaMemsetAsync(hm, 0, ldj * n * sizeof(double), h->stream));
            }
            LAUNCHED(dgemm_dmma_launch(0, P.nvar, P.X, P.nvar, 1.0, Jt, T.ld, 0, dpsi, T.ld, 0, 0.0, hpsi, T.ld, 0, 1, h->stream));
            LAUNCHED(dgemm_dmma_launch(0, P.nvar, P.nvar, P.nvar, 1.0, Jt, T.ld, 0, JtT, T.ld, 0, 0.0, hm, T.ld, 0, 1, h->stream));
        }
        h->factor_valid = true;
    }
    T.Dpsi = use_dpsi ? dpsi : nullptr;
    T.Hpsi = pform ? hpsi : nullptr;
    T.Hm = pform ? hm : nullptr;
    T.Qs = pform ? P.Q : nullptr;
    T.nx = P.nx; T.X = P.X;
    T.Phi = DArr{ P.Phi, (long long)P.X * P.nx };
    T.Gs = DArr{ P.Gs, (long long)P.N * P.nx * P.nu };
    CU(cudaMemsetAsync(counter, 0, 2 * sizeof(int), h->stream));
    for (int k = 0; k < P.nfam; ++k) {
        T.fam[k].EGx = P.fam[k].EGx; T.fam[k].sEGx = P.fam[k].sEGx;
        T.fam[k].E = P.fam[k].hasE ? P.fam[k].E : DArr{ nullptr, 0 };
        T.fam[k].G = P.fam[k].hasG ? P.fam[k].G : DArr{ nullptr, 0 };
    }
    const long long nn = (long long)(ldj * n);
    T.Jt = DArr{ Jt, P.sQ ? nn : 0 };
    T.JtT = DArr{ JtT, P.sQ ? nn : 0 };
    T.pd = pd; T.pd_stride = P.sQ ? 1 : 0;
    T.c = DArr{ P.c, (long long)n };
    T.Aeq = DArr{ nullptr, 0 }; T.Aineq = DArr{ nullptr, 0 };
    T.beq = DArr{ P.meq ? P.beq : nullptr, P.meq };
    T.bineq = DArr{ P.mineq ? P.bineq : nullptr, P.mineq };
    T.lb = DArr{ P.lb, (long long)n };
    T.ub = DArr{ P.ub, (long long)n };
    T.x = x; T.status = status; T.iters = iters; T.nact = nact; T.iact = iact;
    T.ws = wsp; T.ws_stride = plan.ws_stride;
    T.counter = counter;
    T.vsmall = h->vsmall;
    T.max_iter = 50 * (P.meq + P.mineq + 2 * P.nvar) + 100;
    h->solver = "gt_factor_kernel + gi_thin_kernel";
    // few waves of instances per resident CTA: the step ends with the slowest instance, so rank the instances by the number
    // of constraints violated at their unconstrained minimiser (one cheap prepass) and start the heaviest first
    T.prekey = nullptr; T.preidx = nullptr; T.order = nullptr;
    T.kheavy = P.batch;
    // warm start (opt-in): a re-solve of the resident build seeds each instance with the rows active at its previous solve
    int* warm_iact = nullptr;
    if (h->warm_start && pform && (rc = ws(h, "warm_iact", size_t(P.batch) * n, &warm_iact))) return rc;
    T.warm = (h->warm_start && pform && h->in_resolve && h->warm_valid) ? warm_iact : nullptr;
    const int slots = plan.cluster > 1 ? plan.grid / plan.cluster : plan.grid; // instances in flight
    const bool lpt = P.batch > slots && (P.batch <= 24 * slots || plan.cluster > 1);
    cudaError_t e;
    if (lpt) {
        int *keys = nullptr, *keys2 = nullptr, *idx = nullptr, *order = nullptr;
        void* tmp = nullptr;
        const size_t tb = gt_sort_temp_bytes(P.batch);
        if ((rc = ws(h, "gt_keys", 4 * size_t(P.batch), &keys))) return rc;
        if ((rc = dev_reserve(h, "gt_sorttmp", tb, &tmp))) return rc;
        keys2 = keys + P.batch; idx = keys + 2 * size_t(P.batch); order = keys + 3 * size_t(P.batch);
        T.prekey = keys; T.preidx = idx;
        e = gt_launch(T, plan, h->stream);
        if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gt_launch (prepass): %s", cudaGetErrorString(e));
        e = gt_sort_launch(keys, keys2, idx, order, P.batch, tmp, tb, h->stream);
        if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gt_sort_launch: %s", cudaGetErrorString(e));
        h->launches += 2; h->call_launches += 2;
        CU(cudaMemsetAsync(counter, 0, 2 * sizeof(int), h->stream));
        T.prekey = nullptr; T.preidx = nullptr; T.order = order;
        // clusters for the head of the longest-first queue only (the heavy tail of the iteration counts)
        if (plan.cluster > 1) T.kheavy = std::max(1, P.batch / 16);
    }
    e = gt_launch(T, plan, h->stream);
    if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gt_launch: %s", cudaGetErrorString(e));
    h->launches += 1; h->call_launches += 1;
    if (warm_iact && iact) {
        CU(cudaMemcpyAsync(warm_iact, iact, size_t(P.batch) * n * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
        h->warm_valid = true;
    }
    return 0;
}

// materialise Aeq / Aineq of the last build if the build skipped them
int ensure_rows(copra_b200_handle* h)
{
    if (h->rows_filled) return 0;
    BuildParams& P = h->bp;
    const size_t Bz = P.batch, nv = P.nvar;
    int rc;
    if ((rc = ws(h, "Aeq", Bz * P.meq * nv, &P.Aeq))) return rc;
    if ((rc = ws(h, "Aineq", Bz * P.mineq * nv, &P.Aineq))) return rc;
    LAUNCHED(k3_fill_rows_launch(P, h->stream));
    h->rows_filled = true;
    return 0;
}

int do_build(copra_b200_handle* h, const copra_b200_problem* p)
{
    h->qp_solved = false;
    Plan pl;
    int rc = make_plan(h, p, pl);
    if (rc) return rc;
    if (p->batch > 65535) return fail(h, COPRA_B200_E_UNSUPPORTED, "batch > 65535 per call: shard the batch (bench.py does)");
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    for (bool& v : h->ev_valid) v = false;
    rc = record(h, 0);
    if (rc) return rc;

    BuildParams& P = h->bp;
    std::memset(&P, 0, sizeof P);
    const int nx = p->nx, nu = p->nu, N = p->N, B = p->batch;
    P.nx = nx; P.nu = nu; P.N = N; P.batch = B;
    P.X = pl.sz.X; P.nU = pl.sz.nU; P.nvar = pl.sz.nvar; P.meq = pl.sz.meq; P.mineq = pl.sz.mineq;
    P.initial_state = p->initial_state ? 1 : 0;
    P.qdiag = (p->flags & COPRA_B200_FLAG_NO_REG) ? 0.0 : 1e-6;
    P.ncost = int(pl.costs.size());
    P.nfam = int(pl.fams.size());
    // The Hessian is a function of A, B and every cost's M, N, w only (p, x0 and the constraints enter c / b): when all of
    // those are shared by the batch it is assembled and factored ONCE (src/costFunctions.cpp:74-75,103-104,150-152,206-208).
    bool q_shared = !p->initial_state && p->A.stride == 0 && p->B.stride == 0 && B > 1;
    for (int i = 0; i < p->ncost && q_shared; ++i) {
        const copra_b200_cost& c = p->costs[i];
        if (c.full_size == 1 || (c.M.ptr && c.M.stride != 0) || (c.N.ptr && c.N.stride != 0) || c.w.stride != 0) q_shared = false;
    }
    P.sQ = q_shared ? 0 : (long long)pl.sz.nvar * pl.sz.nvar;

    // selector matrices + line indices for TrajectoryBound families (tiny, shared by all instances)
    std::vector<double> sel;
    std::vector<int> lines;
    std::vector<size_t> sel_off(pl.fams.size(), 0), line_off(pl.fams.size(), 0);
    for (size_t k = 0; k < pl.fams.size(); ++k) {
        const auto& f = pl.fams[k];
        if (f.which == 0) continue;
        sel_off[k] = sel.size();
        line_off[k] = lines.size();
        if (!f.gather) sel.resize(sel.size() + size_t(f.rows) * nx, 0.0);
        for (int l = 0; l < f.rows; ++l) {
            if (!f.gather) sel[sel_off[k] + l + size_t(f.lines[l]) * f.rows] = 1.0;
            lines.push_back(f.lines[l]);
        }
    }
    double* d_sel = nullptr;
    int* d_lines = nullptr;
    if (!lines.empty()) {
        rc = ws(h, "sel", sel.size(), &d_sel); if (rc) return rc;
        rc = ws(h, "lines", lines.size(), &d_lines); if (rc) return rc;
        if (sel != h->sel_host || lines != h->lines_host) {
            CU(cudaStreamSynchronize(h->stream)); // previous kernels may still read the old selectors
            h->sel_host = sel;
            h->lines_host = lines;
            CU(cudaMemcpyAsync(d_sel, h->sel_host.data(), sel.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
            CU(cudaMemcpyAsync(d_lines, h->lines_host.data(), lines.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
            CU(cudaStreamSynchronize(h->stream));
        }
    }

    // parameters
    Upload U;
    U.add(p->A, size_t(nx) * nx, &P.A);
    U.add(p->B, size_t(nx) * nu, &P.B);
    U.add(p->d, nx, &P.d);
    if (p->initial_state) {
        U.add(p->R, size_t(nx) * nx, &P.R);
        U.add(p->r, nx, &P.r);
        U.add(p->x0lb, nx, &P.x0lb);
        U.add(p->x0ub, nx, &P.x0ub);
    }
    for (int i = 0; i < P.ncost; ++i) {
        const copra_b200_cost& c = p->costs[i];
        CostFam& F = P.cost[i];
        F.rows = c.rows; F.i0 = pl.costs[i].i0; F.i1 = pl.costs[i].i1; F.hasM = pl.costs[i].hasM; F.hasN = pl.costs[i].hasN;
        F.dense = pl.costs[i].dense;
        F.pstep = pl.costs[i].pstep;
        if (F.hasM) U.add(c.M, size_t(c.rows) * (F.dense ? pl.sz.X : nx), &F.M);
        if (F.hasN) U.add(c.N, size_t(c.rows) * (F.dense ? pl.sz.nU : nu), &F.N);
        U.add(c.w, c.rows, &F.w);
    }
    for (int k = 0; k < P.nfam; ++k) {
        const auto& f = pl.fams[k];
        const copra_b200_constraint& c = p->cstrs[f.cstr];
        CstrFam& F = P.fam[k];
        F.rows = f.rows; F.i0 = f.i0; F.i1 = f.i1; F.hasE = f.hasE; F.hasG = f.hasG; F.is_eq = f.is_eq; F.row_off = f.row_off;
        F.dense = f.dense; F.gather = f.gather; F.fstep = f.fstep;
        F.fidx = nullptr;
        if (f.which == 0) {
            if (f.hasE) U.add(c.E, size_t(c.rows) * (f.dense ? pl.sz.X : nx), &F.E);
            if (f.hasG) U.add(c.G, size_t(c.rows) * (f.dense ? pl.sz.nU : nu), &F.G);
        }
    }
    BoundArrs ba;
    add_vectors(U, p, pl, P, ba);
    rc = run_upload(h, U, B, p->memory, "params");
    if (rc) return rc;
    for (int k = 0; k < P.nfam; ++k) {
        const auto& f = pl.fams[k];
        if (f.which == 0) continue;
        CstrFam& F = P.fam[k];
        F.E.p = f.gather ? nullptr : d_sel + sel_off[k];
        F.E.s = 0;
        F.fidx = d_lines + line_off[k];
    }
    bind_bounds(pl, P, ba);
    rc = record(h, 1);
    if (rc) return rc;

    // workspace
    const size_t X = P.X, nU = P.nU, nv = P.nvar, meq = P.meq, m = P.mineq, Bz = B;
    if ((rc = ws(h, "Phi", Bz * X * nx, &P.Phi))) return rc;
    if ((rc = ws(h, "Gs", Bz * size_t(N) * nx * nu, &P.Gs))) return rc;
    if ((rc = ws(h, "xi", Bz * X, &P.xi))) return rc;
    if ((rc = ws(h, "Q", (P.sQ ? Bz : size_t(1)) * nv * nv, &P.Q))) return rc;
    if ((rc = ws(h, "c", Bz * nv, &P.c))) return rc;
    plan_thin(h);
    P.skip_rows = h->use_thin ? 1 : 0; // the structured solver evaluates the rows from the E A^k B tables
    P.Aeq = P.Aineq = nullptr;
    if (!P.skip_rows && (rc = ws(h, "Aeq", Bz * meq * nv, &P.Aeq))) return rc;
    if ((rc = ws(h, "beq", Bz * meq, &P.beq))) return rc;
    if (!P.skip_rows && (rc = ws(h, "Aineq", Bz * m * nv, &P.Aineq))) return rc;
    if ((rc = ws(h, "bineq", Bz * m, &P.bineq))) return rc;
    if ((rc = ws(h, "lb", Bz * nv, &P.lb))) return rc;
    if ((rc = ws(h, "ub", Bz * nv, &P.ub))) return rc;
    if ((rc = ws(h, "Yeq", Bz * meq * nx, &P.Yeq))) return rc;
    if ((rc = ws(h, "zeq", Bz * meq, &P.zeq))) return rc;
    if ((rc = ws(h, "Yin", Bz * m * nx, &P.Yin))) return rc;
    if ((rc = ws(h, "zin", Bz * m, &P.zin))) return rc;
    for (int i = 0; i < P.ncost; ++i) {
        CostFam& F = P.cost[i];
        const size_t r = F.rows, ns = F.i1 - F.i0;
        char nm[32];
        F.sMGx = r * nu * (N + 1); F.sMPhi = r * nx * ns; F.sres = r * ns; F.sE = size_t(nx) * nU; F.sf = nU;
        // E = (M Phi)' W (M Psi + N) does not depend on p, x0 or d: one copy for the batch when A, B, M, N, w are shared
        // (src/costFunctions.cpp:77,105,210) -- the per-instance part of the assembly is f alone
        const bool e_shared = !F.dense && P.A.s == 0 && P.B.s == 0 && (!F.hasM || F.M.s == 0) && (!F.hasN || F.N.s == 0) && F.w.s == 0;
        if (e_shared) F.sE = 0;
        snprintf(nm, sizeof nm, "MGx%d", i); if ((rc = ws(h, nm, Bz * F.sMGx, &F.MGx))) return rc;
        snprintf(nm, sizeof nm, "MPhi%d", i); if ((rc = ws(h, nm, Bz * F.sMPhi, &F.MPhi))) return rc;
        snprintf(nm, sizeof nm, "res%d", i); if ((rc = ws(h, nm, Bz * F.sres, &F.res))) return rc;
        snprintf(nm, sizeof nm, "Ec%d", i); if ((rc = ws(h, nm, (F.sE ? Bz : size_t(1)) * size_t(nx) * nU, &F.E))) return rc;
        snprintf(nm, sizeof nm, "fc%d", i); if ((rc = ws(h, nm, Bz * F.sf, &F.f))) return rc;
        F.T = F.WT = nullptr; F.sT = 0;
        if (F.dense) {
            F.sT = (long long)(r * nU);
            snprintf(nm, sizeof nm, "Tc%d", i); if ((rc = ws(h, nm, Bz * F.sT, &F.T))) return rc;
            snprintf(nm, sizeof nm, "WTc%d", i); if ((rc = ws(h, nm, Bz * F.sT, &F.WT))) return rc;
        }
    }
    {
        bool need_psi = false;
        for (int i = 0; i < P.ncost; ++i) need_psi |= P.cost[i].dense && P.cost[i].hasM;
        for (int k = 0; k < P.nfam; ++k) need_psi |= P.fam[k].dense && P.fam[k].hasE;
        P.PsiFull = nullptr;
        if (need_psi && (rc = ws(h, "Psi", Bz * X * nU, &P.PsiFull))) return rc;
    }
    for (int k = 0; k < P.nfam; ++k) {
        CstrFam& F = P.fam[k];
        char nm[32];
        F.sEGx = size_t(F.rows) * nu * (N + 1);
        snprintf(nm, sizeof nm, "EGx%d", k);
        if ((rc = ws(h, nm, Bz * F.sEGx, &F.EGx))) return rc;
    }
    double* schur = nullptr;
    long long schur_stride = 0;
    if (P.initial_state) {
        schur_stride = (long long)odd_ld(P.nU) * P.nU;
        if ((rc = ws(h, "schur", size_t(h->sms) * 8 * schur_stride, &schur))) return rc;
    }

    // (a single fused K1..K4 kernel, one CTA per instance, was measured at 0.85 ms vs 0.44 ms for these staged launches
    // on C2: the staged kernels expose far more parallelism per phase, so they stay)
    LAUNCHED(k1_condense_launch(P, h->stream));
    if ((rc = record(h, 2))) return rc;
    LAUNCHED(k2k4_assemble_launch(P, schur, schur_stride, h->sms, h->smem_optin, h->stream));
    if ((rc = record(h, 3))) return rc;
    h->sz = pl.sz;
    h->shape = shape_key(p, pl);
    h->cost_len.clear();
    for (int i = 0; i < P.ncost; ++i) h->cost_len.push_back(p->costs[i].rows * pl.costs[i].vsteps);
    h->cstr_len.clear();
    for (int i = 0; i < p->ncstr; ++i) h->cstr_len.push_back(p->cstrs[i].rows * pl.cvsteps[i]);
    h->fam_cstr.clear();
    h->fam_which.clear();
    for (const auto& f : pl.fams) { h->fam_cstr.push_back(f.cstr); h->fam_which.push_back(f.which); }
    h->bound_cstr = pl.bound_cstr;
    h->built = true;
    h->solved = false;
    h->factor_valid = false;
    h->vjp_factor_valid = false;
    h->warm_valid = false;
    h->gs_j_valid = false;
    h->rows_filled = !P.skip_rows;
    return 0;
}

int do_solve(copra_b200_handle* h, const copra_b200_results* r)
{
    h->qp_solved = false;
    if (!h->built) return fail(h, COPRA_B200_E_STATE, "copra_b200_lmpc_solve called before a successful build");
    h->solved = false;
    const BuildParams& P = h->bp;
    const size_t B = P.batch, nv = P.nvar;
    int rc;
    double *x = nullptr, *control = nullptr, *traj = nullptr;
    int *status = nullptr, *iters = nullptr, *nact = nullptr, *iact = nullptr;
    const bool devres = r && r->memory == COPRA_B200_DEVICE;
    if ((rc = ws(h, "res_x", B * nv, &x))) return rc;
    if ((rc = ws(h, "res_control", B * P.nU, &control))) return rc;
    if ((rc = ws(h, "res_traj", B * P.X, &traj))) return rc;
    if ((rc = ws(h, "res_status", B, &status))) return rc;
    if ((rc = ws(h, "res_iters", 2 * B, &iters))) return rc;
    if ((rc = ws(h, "res_nact", B, &nact))) return rc;
    if ((rc = ws(h, "res_iact", B * nv, &iact))) return rc;
    double* ws_x = x;
    int *ws_status = status, *ws_nact = nact, *ws_iact = iact;
    if (devres) { // write straight into the caller's device buffers where given
        if (r->x) x = r->x;
        if (r->control) control = r->control;
        if (r->trajectory) traj = r->trajectory;
        if (r->status) status = r->status;
        if (r->iters) iters = r->iters;
        if (r->nact) nact = r->nact;
        if (r->iact) iact = r->iact;
    }
    GiBatch G{};
    G.n = P.nvar; G.meq = P.meq; G.m = P.mineq; G.batch = P.batch;
    G.Q = DArr{ P.Q, P.sQ };
    G.c = DArr{ P.c, (long long)nv };
    G.Aeq = DArr{ P.meq ? P.Aeq : nullptr, (long long)(size_t(P.meq) * nv) };
    G.beq = DArr{ P.meq ? P.beq : nullptr, P.meq };
    G.Aineq = DArr{ P.mineq ? P.Aineq : nullptr, (long long)(size_t(P.mineq) * nv) };
    G.bineq = DArr{ P.mineq ? P.bineq : nullptr, P.mineq };
    G.lb = DArr{ P.lb, (long long)nv };
    G.ub = DArr{ P.ub, (long long)nv };
    G.x = x; G.status = status; G.iters = iters; G.nact = nact; G.iact = iact;
    if (h->use_thin) {
        if ((rc = run_gt(h, x, status, iters, nact, iact))) return rc;
    } else {
        if ((rc = ensure_rows(h))) return rc;
        G.Aeq.p = P.meq ? h->bp.Aeq : nullptr;
        G.Aineq.p = P.mineq ? h->bp.Aineq : nullptr;
        h->lmpc_solve_active = true;
        rc = run_gi(h, G);
        h->lmpc_solve_active = false;
        if (rc) return rc;
    }
    if ((rc = record(h, 4))) return rc;
    // the solution and the active sets of this solve stay in the workspace for copra_b200_lmpc_vjp
    if (x != ws_x) CU(cudaMemcpyAsync(ws_x, x, B * nv * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    if (status != ws_status) CU(cudaMemcpyAsync(ws_status, status, B * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
    if (nact != ws_nact) CU(cudaMemcpyAsync(ws_nact, nact, B * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
    if (iact != ws_iact) CU(cudaMemcpyAsync(ws_iact, iact, B * nv * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
    const bool want_ct = !r || r->control || r->trajectory;
    if (want_ct) LAUNCHED(k7_results_launch(P, x, control, traj, h->stream));
    if ((rc = record(h, 5))) return rc;
    if (r && !devres) {
        Download D;
        D.add(x, r->x, B * nv * sizeof(double));
        D.add(control, r->control, B * P.nU * sizeof(double));
        D.add(traj, r->trajectory, B * P.X * sizeof(double));
        D.add(status, r->status, B * sizeof(int));
        D.add(iters, r->iters, 2 * B * sizeof(int));
        D.add(nact, r->nact, B * sizeof(int));
        D.add(iact, r->iact, B * nv * sizeof(int));
        if ((rc = run_download(h, D, COPRA_B200_HOST))) return rc;
    }
    if ((rc = record(h, 6))) return rc;
    h->solved = true;
    return 0;
}

// Where the K8 / K9 core finds R^-1 (ld gt_even(n)) of the Hessian of a chunk of instances: Jt of the chunk's first instance,
// sJ doubles apart (0 = one factor for the batch), and the positive-definiteness flags of the whole batch, qpd_stride apart
struct SensFactor {
    const double* Jt;
    long long sJ;
    const int* qpd;
    int qpd_stride;
};

// R^-1 of the resident build's Hessian(s) for K8 / K9 (ld gt_even(n); one per instance when P.sQ, else one for the batch):
// the thin solver's resident factor, else one factorisation kept until the next build
int sens_factor(copra_b200_handle* h, const double** Jt, const int** qpd)
{
    const BuildParams& P = h->bp;
    const size_t n = P.nvar, count = P.sQ ? size_t(P.batch) : 1;
    const int ldj = gt_even(int(n));
    int rc;
    if (h->use_thin && h->factor_valid) {
        *Jt = static_cast<const double*>(h->dev["gt_Jt"].p);
        *qpd = static_cast<const int*>(h->dev["gt_pd"].p);
        return 0;
    }
    double *J = nullptr, *JT = nullptr;
    int* pd = nullptr;
    if ((rc = ws(h, "vjp_Jt", count * ldj * n, &J))) return rc;
    if ((rc = ws(h, "vjp_JtT", count * ldj * n, &JT))) return rc;
    if ((rc = ws(h, "vjp_pd", count, &pd))) return rc;
    if (!h->vjp_factor_valid) {
        cudaError_t e = gt_factor_launch(DArr{ P.Q, P.sQ }, int(n), ldj, int(count), J, JT, pd, h->plan_sms, h->stream);
        if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gt_factor_launch: %s", cudaGetErrorString(e));
        h->launches += 1; h->call_launches += 1;
        h->vjp_factor_valid = true;
    }
    *Jt = J;
    *qpd = pd;
    return 0;
}

// The active-set KKT solve of K8 / K9 for the last solve (n variables, `batch` instances; res_status / res_nact / res_iact
// hold its status and active sets), with k right-hand sides per instance.  The batch is processed in chunks whose slab, Y and
// Gram workspace, plus `factor_per` doubles per instance for a factor made per chunk, stay under kSensWsBytes, each padded to
// its own largest active set.  `factor(b0, nb, F)` provides the chunk's Hessian factor, launching what it needs; `first(nb)`
// writes a chunk's slab and rhs (the right-hand sides), `last(nb)` reads its V (and rhs = M); both launch one kernel.
constexpr size_t kSensWsBytes = size_t(1) << 30;

template <class Factor, class First, class Last>
int sens_run(copra_b200_handle* h, SensChunk& S, int n_, int batch, int k, size_t factor_per, Factor factor, First first, Last last)
{
    const size_t B = batch, n = n_, K = size_t(k);
    int rc;
    int *status = nullptr, *nact = nullptr, *iact = nullptr;
    if ((rc = ws(h, "res_status", B, &status))) return rc;
    if ((rc = ws(h, "res_nact", B, &nact))) return rc;
    if ((rc = ws(h, "res_iact", B * n, &iact))) return rc;
    // the largest active set of the solved instances sizes the workspace, each chunk uses its own largest
    std::vector<int> hs(B), hn(B);
    CU(cudaMemcpyAsync(hs.data(), status, B * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(hn.data(), nact, B * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    auto widest = [&](size_t lo, size_t hi) {
        int w = 0;
        for (size_t b = lo; b < hi; ++b) if (hs[b] == 0) w = std::max(w, hn[b]);
        return w;
    };
    const int nm = widest(0, B);
    const int ldj = gt_even(int(n));
    // chunked workspace
    const size_t lds = size_t(ldj), mk = size_t(nm) + K, ldg = size_t(gt_even(nm));
    const size_t per = 2 * lds * mk + mk * mk + size_t(nm) * nm + 2 * ldg * nm + size_t(nm) * K + 2 * lds * K + 1 + factor_per;
    const int chunk = int(std::max<size_t>(1, std::min<size_t>(B, kSensWsBytes / (per * sizeof(double)))));
    S.n = int(n); S.k = k; S.lds = int(lds); S.ldy = int(lds);
    S.status = status; S.nact = nact; S.iact = iact;
    double* GJT = nullptr;
    const size_t C = size_t(chunk);
    if ((rc = ws(h, "vjp_slab", C * lds * mk, &S.slab))) return rc;
    if ((rc = ws(h, "vjp_Y", C * lds * mk, &S.Y))) return rc;
    if ((rc = ws(h, "vjp_Gf", C * mk * mk, &S.Gf))) return rc;
    if ((rc = ws(h, "vjp_Gq", C * nm * nm, &S.Gq))) return rc;
    if ((rc = ws(h, "vjp_GJ", C * ldg * nm, const_cast<double**>(&S.GJ)))) return rc;
    if ((rc = ws(h, "vjp_GJT", C * ldg * nm, &GJT))) return rc;
    if ((rc = ws(h, "vjp_gpd", C, const_cast<int**>(&S.gpd)))) return rc;
    if ((rc = ws(h, "vjp_rhs", C * nm * K, &S.rhs))) return rc;
    if ((rc = ws(h, "vjp_W", C * lds * K, &S.W))) return rc;
    if ((rc = ws(h, "vjp_V", C * lds * K, &S.V))) return rc;
    const int N_ = int(n), L = int(lds);
    for (int b0 = 0; b0 < batch; b0 += chunk) {
        const int nb = std::min(chunk, batch - b0);
        const int nm = widest(size_t(b0), size_t(b0) + nb), MK = nm + k;
        SensFactor F{};
        if ((rc = factor(b0, nb, F))) return rc;
        const double* Jt = F.Jt;
        const long long sJ = F.sJ;
        S.qpd = F.qpd; S.qpd_stride = F.qpd_stride;
        S.b0 = b0; S.nm = nm; S.ldg = gt_even(nm);
        LAUNCHED(first(nb));
        // Y = Jt' slab: one GEMM over the chunk for a shared factor
        if (sJ == 0) LAUNCHED(dgemm_dmma_launch(1, N_, nb * MK, N_, 1.0, Jt, ldj, 0, S.slab, L, 0, 0.0, S.Y, L, 0, 1, h->stream));
        else LAUNCHED(dgemm_dmma_launch(1, N_, MK, N_, 1.0, Jt, ldj, sJ, S.slab, L, (long long)L * MK, 0.0, S.Y, L,
            (long long)L * MK, nb, h->stream));
        if (nm > 0) {
            LAUNCHED(dgemm_dmma_launch(1, MK, MK, N_, 1.0, S.Y, L, (long long)L * MK, S.Y, L, (long long)L * MK, 0.0, S.Gf, MK,
                (long long)MK * MK, nb, h->stream));
            LAUNCHED(sens_gram_launch(S, nb, h->stream));
            cudaError_t e = gt_factor_launch(DArr{ S.Gq, (long long)nm * nm }, nm, S.ldg, nb, const_cast<double*>(S.GJ), GJT,
                const_cast<int*>(S.gpd), h->plan_sms, h->stream);
            if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gt_factor_launch: %s", cudaGetErrorString(e));
            h->launches += 1; h->call_launches += 1;
        }
        LAUNCHED(sens_solve_launch(S, nb, h->stream));
        // V = Jt W
        if (sJ == 0) LAUNCHED(dgemm_dmma_launch(0, N_, nb * k, N_, 1.0, Jt, ldj, 0, S.W, L, 0, 0.0, S.V, L, 0, 1, h->stream));
        else LAUNCHED(dgemm_dmma_launch(0, N_, k, N_, 1.0, Jt, ldj, sJ, S.W, L, (long long)L * k, 0.0, S.V, L,
            (long long)L * k, nb, h->stream));
        LAUNCHED(last(nb));
    }
    return 0;
}

// the factor source of the resident LMPC build: sens_factor's, made once and kept until the next build
int lmpc_factor(copra_b200_handle* h, int b0, SensFactor& F)
{
    const BuildParams& P = h->bp;
    const double* Jt = nullptr;
    int rc = sens_factor(h, &Jt, &F.qpd);
    if (rc) return rc;
    F.sJ = P.sQ ? (long long)gt_even(P.nvar) * P.nvar : 0;
    F.Jt = Jt + b0 * F.sJ;
    F.qpd_stride = P.sQ ? 1 : 0;
    return 0;
}

// the gradients a VJP writes: the caller's device buffers, or (HOST) one workspace block downloaded by download_outputs;
// every wanted one is zeroed on the stream first (the kernels write only the entries they own)
struct OutItem { double* host; double** dev; size_t len; };

int bind_outputs(copra_b200_handle* h, std::vector<OutItem>& items, size_t B, int memory)
{
    int rc;
    size_t total = 0;
    for (auto& it : items) if (it.host) total += it.len * B;
    double* oblk = nullptr;
    if (memory == COPRA_B200_HOST && total && (rc = ws(h, "vjp_out", total, &oblk))) return rc;
    total = 0;
    for (auto& it : items) {
        if (!it.host) continue;
        *it.dev = memory == COPRA_B200_HOST ? oblk + total : it.host;
        total += it.len * B;
        if (memory == COPRA_B200_DEVICE) CU(cudaMemsetAsync(*it.dev, 0, it.len * B * sizeof(double), h->stream));
    }
    if (oblk) CU(cudaMemsetAsync(oblk, 0, total * sizeof(double), h->stream));
    return 0;
}

int download_outputs(copra_b200_handle* h, const std::vector<OutItem>& items, size_t B, int memory)
{
    if (memory != COPRA_B200_HOST) return 0;
    Download D;
    for (auto& it : items) if (it.host) D.add(*it.dev, it.host, it.len * B * sizeof(double));
    return run_download(h, D, COPRA_B200_HOST);
}

// K8 for the last solve (copra_b200_lmpc_vjp, _vjp_costs, _vjp_model, _vjp_initial_state): the outputs are zeroed first and
// k8_adjoint only writes the entries it owns; with `costs`, k8_cost_grad follows k8_adjoint on each chunk and writes the cost
// gradients; with `model`, the KKT solve takes the forward solve as a second right-hand side (its multipliers) and
// k8_model_grad follows them and writes the model gradients.  `init` (initial-state builds) adds R, r, x0lb and x0ub to
// k8_adjoint's outputs.
int do_vjp(copra_b200_handle* h, const double* dcontrol, const double* dtraj, int memory, const copra_b200_vjp_out* out,
    const copra_b200_vjp_cost_out* costs, const copra_b200_vjp_model_out* model, const copra_b200_vjp_initial_out* init = nullptr)
{
    const BuildParams& P = h->bp;
    const size_t B = P.batch, nx = P.nx, nu = P.nu;
    int rc;
    static const copra_b200_vjp_out none{};
    if (!out) out = &none;
    // inputs
    const double *dc = dcontrol, *dt = dtraj;
    if (memory == COPRA_B200_HOST && (dcontrol || dtraj)) {
        double* in = nullptr;
        if ((rc = ws(h, "vjp_in", B * (P.nU + P.X), &in))) return rc;
        if (dcontrol) CU(cudaMemcpyAsync(in, dcontrol, B * P.nU * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        if (dtraj) CU(cudaMemcpyAsync(in + B * P.nU, dtraj, B * P.X * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        dc = dcontrol ? in : nullptr;
        dt = dtraj ? in + B * P.nU : nullptr;
    }
    // outputs: the caller's device buffers, or one workspace block downloaded at the end
    VjpParams V{};
    std::vector<OutItem> items;
    items.push_back({ out->x0, &V.dx0, nx });
    for (int ci = 0; ci < P.ncost; ++ci) {
        V.plen[ci] = h->cost_len[ci];
        items.push_back({ out->p ? out->p[ci] : nullptr, &V.dp[ci], size_t(h->cost_len[ci]) });
    }
    for (int fi = 0; fi < P.nfam; ++fi) {
        const int c = h->fam_cstr[fi], which = h->fam_which[fi];
        double* const* arr = which == 0 ? out->f : (which == 1 ? out->lower : out->upper);
        V.flen[fi] = h->cstr_len[c];
        items.push_back({ arr ? arr[c] : nullptr, &V.df[fi], size_t(h->cstr_len[c]) });
    }
    if (h->bound_cstr >= 0) {
        V.cblen = h->cstr_len[h->bound_cstr];
        items.push_back({ out->lower ? out->lower[h->bound_cstr] : nullptr, &V.dlower, size_t(V.cblen) });
        items.push_back({ out->upper ? out->upper[h->bound_cstr] : nullptr, &V.dupper, size_t(V.cblen) });
    }
    bool want_costs = false;
    if (costs) {
        for (int ci = 0; ci < P.ncost; ++ci) {
            const size_t r = P.cost[ci].rows;
            items.push_back({ costs->w ? costs->w[ci] : nullptr, &V.dw[ci], r });
            items.push_back({ costs->M ? costs->M[ci] : nullptr, &V.dM[ci], r * nx });
            items.push_back({ costs->N ? costs->N[ci] : nullptr, &V.dN[ci], r * nu });
            want_costs |= (costs->w && costs->w[ci]) || (costs->M && costs->M[ci]) || (costs->N && costs->N[ci]);
        }
    }
    bool want_model = false;
    if (model) {
        items.push_back({ model->A, &V.dA, nx * nx });
        items.push_back({ model->B, &V.dB, nx * nu });
        items.push_back({ model->d, &V.dd, nx });
        want_model = model->A || model->B || model->d;
        for (int fi = 0; fi < P.nfam; ++fi) {
            if (h->fam_which[fi] != 0) continue; // a trajectory bound's E is the engine's selector
            const int c = h->fam_cstr[fi];
            const size_t r = P.fam[fi].rows;
            double* E = model->E ? model->E[c] : nullptr;
            double* G = model->G ? model->G[c] : nullptr;
            items.push_back({ E, &V.dE[fi], r * nx });
            items.push_back({ G, &V.dG[fi], r * nu });
            want_model |= E || G;
        }
    }
    if (init) {
        items.push_back({ init->R, &V.dR, nx * nx });
        items.push_back({ init->r, &V.dr, nx });
        items.push_back({ init->x0lb, &V.dx0lb, nx });
        items.push_back({ init->x0ub, &V.dx0ub, nx });
    }
    const bool want_x = want_costs || want_model || (init && init->R);
    if (want_x && (rc = ws(h, "res_x", B * P.nvar, &V.U))) return rc;
    if ((rc = bind_outputs(h, items, B, memory))) return rc;
    V.dcontrol = dc; V.sdc = P.nU; V.dtraj = dt; V.sdt = P.X;
    rc = sens_run(h, V, P.nvar, P.batch, want_model ? 2 : 1, 0, [&](int b0, int, SensFactor& F) { return lmpc_factor(h, b0, F); },
        [&](int nb) { return k8_gather_launch(P, V, nb, h->stream); },
        [&](int nb) {
            int n = k8_adjoint_launch(P, V, nb, h->stream);
            if (n < 0) return n;
            if (want_costs) {
                const int n2 = k8_cost_grad_launch(P, V, nb, h->stream);
                if (n2 < 0) return n2;
                n += n2;
            }
            if (want_model) {
                const int n3 = k8_model_grad_launch(P, V, nb, h->stream);
                if (n3 < 0) return n3;
                n += n3;
            }
            return n;
        });
    if (rc) return rc;
    return download_outputs(h, items, B, memory);
}

// K9 for the last solve (copra_b200_lmpc_jvp, copra_b200_lmpc_feedback_gain, copra_b200_lmpc_jvp_initial_state): k tangent
// directions described by `in` (and, initial-state builds, `init`), or (gain) the columns of the identity on x0.  k9_output
// writes every entry of the first ru rows of dU and the first rx rows of dtrajectory of each direction (zeros for an instance
// whose status is not 0).
int do_jvp(copra_b200_handle* h, const copra_b200_jvp_in* in, int k, bool gain, int memory, double* dcontrol, int ru,
    double* dtraj, int rx, const copra_b200_jvp_initial_in* init = nullptr)
{
    const BuildParams& P = h->bp;
    const size_t B = P.batch, nx = P.nx, K = size_t(k);
    int rc;
    JvpParams J{};
    J.gain = gain ? 1 : 0;
    // tangents: the caller's device arrays, or HOST arrays packed into the staging buffer and uploaded in one copy
    Upload U;
    DArr tx0{}, tp[kMaxCost]{}, tf[kMaxFam]{}, tlo{}, tup{}, tR{}, tr{}, tx0lb{}, tx0ub{};
    auto add = [&](const double* a, size_t len, DArr* dst) { U.add(copra_b200_array{ a, (long long)(len * K) }, len * K, dst); };
    if (in) {
        add(in->x0, nx, &tx0);
        for (int ci = 0; ci < P.ncost; ++ci) {
            J.plen[ci] = h->cost_len[ci];
            add(in->p ? in->p[ci] : nullptr, size_t(h->cost_len[ci]), &tp[ci]);
        }
        for (int fi = 0; fi < P.nfam; ++fi) {
            const int c = h->fam_cstr[fi], which = h->fam_which[fi];
            const double* const* arr = which == 0 ? in->f : (which == 1 ? in->lower : in->upper);
            J.flen[fi] = h->cstr_len[c];
            add(arr ? arr[c] : nullptr, size_t(h->cstr_len[c]), &tf[fi]);
        }
        if (h->bound_cstr >= 0) {
            J.cblen = h->cstr_len[h->bound_cstr];
            add(in->lower ? in->lower[h->bound_cstr] : nullptr, size_t(J.cblen), &tlo);
            add(in->upper ? in->upper[h->bound_cstr] : nullptr, size_t(J.cblen), &tup);
        }
    }
    if (init) {
        add(init->R, nx * nx, &tR);
        add(init->r, nx, &tr);
        add(init->x0lb, nx, &tx0lb);
        add(init->x0ub, nx, &tx0ub);
    }
    if ((rc = run_upload(h, U, P.batch, memory, "jvp_in"))) return rc;
    J.tR = tR.p; J.tr = tr.p; J.tx0lb = tx0lb.p; J.tx0ub = tx0ub.p;
    if (J.tR && (rc = ws(h, "res_x", B * P.nvar, const_cast<double**>(&J.x)))) return rc;
    J.tx0 = tx0.p;
    for (int ci = 0; ci < P.ncost; ++ci) J.tp[ci] = tp[ci].p;
    for (int fi = 0; fi < P.nfam; ++fi) J.tf[fi] = tf[fi].p;
    J.tlower = tlo.p;
    J.tupper = tup.p;
    // outputs: the caller's device buffers, or one workspace block downloaded at the end
    J.ru = ru; J.rx = rx;
    J.dcontrol = dcontrol; J.dtraj = dtraj;
    if (memory == COPRA_B200_HOST && (dcontrol || dtraj)) {
        double* oblk = nullptr;
        if ((rc = ws(h, "jvp_out", B * (size_t(ru) + size_t(rx)) * K, &oblk))) return rc;
        J.dcontrol = dcontrol ? oblk : nullptr;
        J.dtraj = dtraj ? oblk + B * size_t(ru) * K : nullptr;
    }
    rc = sens_run(h, J, P.nvar, P.batch, k, 0, [&](int b0, int, SensFactor& F) { return lmpc_factor(h, b0, F); },
        [&](int nb) { return k9_tangent_launch(P, J, nb, h->stream); },
        [&](int nb) { return k9_output_launch(P, J, nb, h->stream); });
    if (rc) return rc;
    if (memory == COPRA_B200_HOST) {
        Download D;
        D.add(J.dcontrol, dcontrol, B * size_t(ru) * K * sizeof(double));
        D.add(J.dtraj, dtraj, B * size_t(rx) * K * sizeof(double));
        if ((rc = run_download(h, D, COPRA_B200_HOST))) return rc;
    }
    return 0;
}

// The factor source of the last raw QP batch for sens_run: R^-1 of its Q in workspace of its own (`prefix`_Jt, _JtT, _pd), so
// the resident LMPC build's factors survive: one factorisation for a stride-0 Q (at the first chunk), else one per chunk
// (counted in the chunk's bytes instead of 2 ld n doubles for the whole batch)
int qp_factor(copra_b200_handle* h, const std::string& prefix, int b0, int nb, SensFactor& F)
{
    const GiBatch& G = h->qp;
    const size_t n = G.n;
    const int ldj = gt_even(G.n);
    const bool shared_q = G.Q.s == 0;
    double *J = nullptr, *JT = nullptr;
    int* pd = nullptr;
    const size_t count = shared_q ? 1 : size_t(nb); // the first chunk is the largest: later ones reuse its workspace
    int rc;
    if ((rc = ws(h, (prefix + "_Jt").c_str(), count * ldj * n, &J))) return rc;
    if ((rc = ws(h, (prefix + "_JtT").c_str(), count * ldj * n, &JT))) return rc;
    if ((rc = ws(h, (prefix + "_pd").c_str(), shared_q ? 1 : size_t(G.batch), &pd))) return rc;
    if (!shared_q || b0 == 0) {
        cudaError_t e = gt_factor_launch(DArr{ G.Q.at(shared_q ? 0 : b0), G.Q.s }, G.n, ldj, int(count), J, JT,
            shared_q ? pd : pd + b0, h->plan_sms, h->stream);
        if (e != cudaSuccess) return fail(h, COPRA_B200_E_CUDA, "gt_factor_launch: %s", cudaGetErrorString(e));
        h->launches += 1; h->call_launches += 1;
    }
    F.Jt = J;
    F.sJ = shared_q ? 0 : (long long)ldj * (long long)n;
    F.qpd = pd;
    F.qpd_stride = shared_q ? 0 : 1;
    return 0;
}

// K8 for the last raw QP batch (copra_b200_qp_vjp): the same KKT core, fed by qp_gather and finished by qp_grad, with the
// factor of Q from qp_factor.  With dAeq / dAineq the forward solve is the second right-hand side (k = 2) and its multipliers
// lambda enter.
int do_qp_vjp(copra_b200_handle* h, const double* dx, int memory, const copra_b200_qp_vjp_out* out)
{
    const GiBatch& G = h->qp;
    const size_t B = G.batch, n = G.n, meq = G.meq, m = G.m;
    const int ldj = gt_even(G.n);
    int rc;
    const double* d = dx;
    if (memory == COPRA_B200_HOST) {
        double* in = nullptr;
        if ((rc = ws(h, "qpv_in", B * n, &in))) return rc;
        CU(cudaMemcpyAsync(in, dx, B * n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        d = in;
    }
    QpVjpParams V{};
    std::vector<OutItem> items{ { out->Q, &V.dQ, n * n }, { out->c, &V.dc, n }, { out->Aeq, &V.dAeq, meq * n },
        { out->beq, &V.dbeq, meq }, { out->Aineq, &V.dAineq, m * n }, { out->bineq, &V.dbineq, m }, { out->lb, &V.dlb, n },
        { out->ub, &V.dub, n } };
    if ((rc = bind_outputs(h, items, B, memory))) return rc;
    V.meq = G.meq; V.m = G.m;
    V.c = G.c; V.Aeq = G.Aeq; V.beq = G.beq; V.Aineq = G.Aineq; V.bineq = G.bineq; V.lb = G.lb; V.ub = G.ub;
    V.dx = d;
    double* x = nullptr;
    if ((rc = ws(h, "res_x", B * n, &x))) return rc;
    V.x = x;
    const bool shared_q = G.Q.s == 0;
    auto factor = [&](int b0, int nb, SensFactor& F) { return qp_factor(h, "qpv", b0, nb, F); };
    const bool want_rows = out->Aeq || out->Aineq;
    rc = sens_run(h, V, G.n, G.batch, want_rows ? 2 : 1, shared_q ? 0 : 2 * size_t(ldj) * n, factor,
        [&](int nb) { return qp_gather_launch(V, nb, h->stream); }, [&](int nb) { return qp_grad_launch(V, nb, h->stream); });
    if (rc) return rc;
    return download_outputs(h, items, B, memory);
}

// K9 for the last raw QP batch (copra_b200_qp_jvp, copra_b200_qp_jacobian): k tangent directions described by `in`, or (in
// == NULL) the columns of the identity on the input `wrt`.  Q's factor comes from qp_factor with workspace of its own.  With
// Aeq / Aineq tangents a k = 1 pass on the forward right-hand side first leaves lambda in qpj_lam (its own chunking, so its
// own factorisation); without them there is one pass.  qp_output writes every entry of dx (n x k per instance).
int do_qp_jvp(copra_b200_handle* h, const copra_b200_qp_jvp_in* in, int k, int wrt, int memory, double* dx)
{
    const GiBatch& G = h->qp;
    const size_t B = G.batch, n = G.n, meq = G.meq, m = G.m, K = size_t(k);
    int rc;
    QpJvpParams J{};
    J.wrt = in ? -1 : wrt;
    // tangents: the caller's device arrays, or HOST arrays packed into the staging buffer and uploaded in one copy
    Upload U;
    if (in) {
        const struct { copra_b200_array a; size_t len; DArr* dst; } t[] = { { in->Q, n * n, &J.tQ }, { in->c, n, &J.tc },
            { in->Aeq, meq * n, &J.tAeq }, { in->beq, meq, &J.tbeq }, { in->Aineq, m * n, &J.tAineq }, { in->bineq, m, &J.tbineq },
            { in->lb, n, &J.tlb }, { in->ub, n, &J.tub } };
        for (const auto& it : t) U.add(it.a, it.len * K, it.dst);
    }
    if ((rc = run_upload(h, U, G.batch, memory, "qpj_in"))) return rc;
    J.meq = G.meq; J.m = G.m;
    J.c = G.c; J.Aeq = G.Aeq; J.beq = G.beq; J.Aineq = G.Aineq; J.bineq = G.bineq; J.lb = G.lb; J.ub = G.ub;
    if ((rc = ws(h, "res_x", B * n, const_cast<double**>(&J.x)))) return rc;
    J.dx = dx;
    if (memory == COPRA_B200_HOST && (rc = ws(h, "qpj_out", B * n * K, &J.dx))) return rc;
    const size_t factor_per = G.Q.s == 0 ? 0 : 2 * size_t(gt_even(G.n)) * n;
    auto factor = [&](int b0, int nb, SensFactor& F) { return qp_factor(h, "qpj", b0, nb, F); };
    if (J.tAeq.p || J.tAineq.p) {
        if ((rc = ws(h, "qpj_lam", B * n, &J.lam))) return rc;
        rc = sens_run(h, J, G.n, G.batch, 1, factor_per, factor, [&](int nb) { return qp_lambda_gather_launch(J, nb, h->stream); },
            [&](int nb) { return qp_lambda_store_launch(J, nb, h->stream); });
        if (rc) return rc;
    }
    rc = sens_run(h, J, G.n, G.batch, k, factor_per, factor, [&](int nb) { return qp_tangent_launch(J, nb, h->stream); },
        [&](int nb) { return qp_output_launch(J, nb, h->stream); });
    if (rc) return rc;
    if (memory == COPRA_B200_HOST) {
        Download D;
        D.add(J.dx, dx, B * n * K * sizeof(double));
        if ((rc = run_download(h, D, COPRA_B200_HOST))) return rc;
    }
    return 0;
}

// the resident build takes its vectors only through the vector part of K2 / K4, which retarget re-runs and the sensitivities
// differentiate: no full-size entry other than the control bound
int full_size_check(copra_b200_handle* h, const char* name)
{
    const BuildParams& P = h->bp;
    for (int i = 0; i < P.ncost; ++i)
        if (P.cost[i].dense) return fail(h, COPRA_B200_E_UNSUPPORTED, "%s: cost %d is a full-size entry (its f comes out of the dense GEMMs)", name, i);
    for (int k = 0; k < P.nfam; ++k)
        if (P.fam[k].dense || P.fam[k].gather)
            return fail(h, COPRA_B200_E_UNSUPPORTED, "%s: a row constraint is a full-size entry (its b comes out of the dense GEMMs)", name);
    return 0;
}

// the same, and LMPC mode
int vector_inputs_check(copra_b200_handle* h, const char* name)
{
    if (h->bp.initial_state) return fail(h, COPRA_B200_E_UNSUPPORTED, "%s is defined for LMPC mode only", name);
    return full_size_check(h, name);
}

// the preconditions of the sensitivities of the last solve (copra_b200_lmpc_vjp, _jvp, _feedback_gain)
int sens_check(copra_b200_handle* h, const char* name)
{
    if (!h->built || !h->solved) return fail(h, COPRA_B200_E_STATE, "copra_b200_%s needs a solve of the resident build on this handle", name);
    return vector_inputs_check(h, name);
}

// the preconditions of the initial-state sensitivities (copra_b200_lmpc_vjp_initial_state, _jvp_initial_state), k right-hand
// sides: a solved initial-state build, R / r / x0lb / x0ub gradients or tangents only for the arrays the build was given, and
// k8_adjoint's and sens_solve's shared memory (the active set has at most nvar rows) within the device's limit
int initial_state_check(copra_b200_handle* h, const char* name, const void* R, const void* r, const void* x0lb, const void* x0ub, int k)
{
    if (!h->built || !h->solved) return fail(h, COPRA_B200_E_STATE, "copra_b200_%s needs a solve of the resident build on this handle", name);
    const BuildParams& P = h->bp;
    if (!P.initial_state)
        return fail(h, COPRA_B200_E_UNSUPPORTED, "%s is defined for initial-state builds; an LMPC-mode build takes copra_b200_lmpc_vjp / "
            "copra_b200_lmpc_jvp", name);
    int rc = full_size_check(h, name);
    if (rc) return rc;
    const struct { const void* want; const void* given; const char* what; } arg[] = {
        { R, P.R.p, "R" }, { r, P.r.p, "r" }, { x0lb, P.x0lb.p, "x0lb" }, { x0ub, P.x0ub.p, "x0ub" } };
    for (const auto& a : arg)
        if (a.want && !a.given)
            return fail(h, COPRA_B200_E_ARG, "%s: the build was not given %s (the reference default is used), it has no sensitivity",
                name, a.what);
    const size_t solve = sizeof(double) * 2 * size_t(std::min(k, 8)) * size_t(P.nvar);
    const size_t need = std::max(k8_adjoint_smem(P), solve);
    if (need > h->smem_optin)
        return fail(h, COPRA_B200_E_UNSUPPORTED, "%s: nvar = %d needs %zu bytes of shared memory per block, the device allows %zu", name,
            P.nvar, need, h->smem_optin);
    return 0;
}

} // namespace

void cb_vjp_lengths(const copra_b200_handle* h, int& nx, std::vector<int>& cost_len, std::vector<int>& cstr_len)
{
    nx = h->bp.nx;
    cost_len = h->cost_len;
    cstr_len = h->cstr_len;
}

void cb_cost_shapes(const copra_b200_handle* h, int& nu, std::vector<int>& rows)
{
    nu = h->bp.nu;
    rows.clear();
    for (int i = 0; i < h->bp.ncost; ++i) rows.push_back(h->bp.cost[i].rows);
}

void cb_cstr_rows(const copra_b200_handle* h, std::vector<int>& rows)
{
    rows.assign(h->cstr_len.size(), 0);
    for (int fi = 0; fi < h->bp.nfam; ++fi)
        if (h->fam_which[fi] == 0) rows[h->fam_cstr[fi]] = h->bp.fam[fi].rows;
}

// ===============================================================================================
extern "C" {

int copra_b200_abi_version(void) { return COPRA_B200_ABI_VERSION; }

int copra_b200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int copra_b200_create(const copra_b200_options* opt, copra_b200_handle** out)
{
    if (!out) return COPRA_B200_E_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return COPRA_B200_E_NOGPU;
    const int dev = opt ? opt->device : 0;
    if (dev < 0 || dev >= n) return COPRA_B200_E_ARG;
    if (cudaSetDevice(dev) != cudaSuccess) return COPRA_B200_E_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return COPRA_B200_E_CUDA;
    if (prop.major < 10) return COPRA_B200_E_NOGPU; // kernels are built for sm_100a only
    copra_b200_handle* h = new copra_b200_handle();
    h->device = dev;
    h->sms = prop.multiProcessorCount;
    h->smem_optin = prop.sharedMemPerBlockOptin;
    h->plan_sms = (opt && opt->sm_limit > 0) ? std::min(opt->sm_limit, h->sms) : h->sms;
    h->small_variant = opt ? opt->small_variant : 0;
    h->vsmall = gi_vsmall();
    if (opt && opt->stream) h->stream = static_cast<cudaStream_t>(opt->stream);
    else {
        if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return COPRA_B200_E_CUDA; }
        h->own_stream = true;
    }
    *out = h;
    return COPRA_B200_OK;
}

void copra_b200_destroy(copra_b200_handle* h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (auto& kv : h->dev) if (kv.second.p) cudaFree(kv.second.p);
    if (h->pin_in.p) cudaFreeHost(h->pin_in.p);
    if (h->pin_out.p) cudaFreeHost(h->pin_out.p);
    for (auto& e : h->ev) if (e) cudaEventDestroy(e);
    if (h->h2d_done) cudaEventDestroy(h->h2d_done);
    if (h->own_stream) cudaStreamDestroy(h->stream);
    delete h;
}

const char* copra_b200_last_error(const copra_b200_handle* h) { return h ? h->err.c_str() : "null handle"; }

int copra_b200_set_stream(copra_b200_handle* h, void* s)
{
    if (!h) return COPRA_B200_E_ARG;
    CU(cudaStreamSynchronize(h->stream));
    if (h->own_stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    h->stream = static_cast<cudaStream_t>(s);
    h->tb_cache.clear();
    return 0;
}

int copra_b200_synchronize(copra_b200_handle* h)
{
    if (!h) return COPRA_B200_E_ARG;
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

long long copra_b200_launch_count(const copra_b200_handle* h) { return h ? h->launches : 0; }

int copra_b200_last_timing(const copra_b200_handle* hc, copra_b200_timing* t)
{
    copra_b200_handle* h = const_cast<copra_b200_handle*>(hc);
    if (!h || !t) return COPRA_B200_E_ARG;
    std::memset(t, 0, sizeof *t);
    CU(cudaStreamSynchronize(h->stream));
    auto span = [&](int a, int b) -> float {
        float ms = 0.f;
        if (h->ev_valid[a] && h->ev_valid[b]) cudaEventElapsedTime(&ms, h->ev[a], h->ev[b]);
        return ms;
    };
    t->h2d_ms = span(0, 1); t->condense_ms = span(1, 2); t->assemble_ms = span(2, 3); t->solve_ms = span(3, 4);
    t->rollout_ms = span(4, 5); t->d2h_ms = span(5, 6); t->total_ms = span(0, 6);
    t->launches = h->call_launches;
    return 0;
}

int copra_b200_dgemm_batch(copra_b200_handle* h, int transA, int M, int N, int K, double alpha, const double* A, int lda,
    long long strideA, const double* B, int ldb, long long strideB, double beta, double* C, int ldc, long long strideC, int batch,
    int memory)
{
    if (!h) return COPRA_B200_E_ARG;
    if (M < 0 || N < 0 || K < 0 || batch <= 0 || !A || !B || !C) return fail(h, COPRA_B200_E_ARG, "bad GEMM arguments");
    const int ar = transA ? K : M, ac = transA ? M : K;
    if (lda < ar || ldb < K || ldc < M) return fail(h, COPRA_B200_E_ARG, "leading dimension too small");
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    const double *dA = A, *dB = B;
    double* dC = C;
    long long sA = strideA, sB = strideB, sC = strideC;
    int rc;
    if (memory == COPRA_B200_HOST) {
        // pack each operand densely (ld == rows) and upload
        const size_t nA = size_t(ar) * ac, nB = size_t(K) * N, nC = size_t(M) * N, Bz = batch;
        std::vector<double> hA(nA * Bz), hB(nB * Bz), hC(nC * Bz);
        for (size_t b = 0; b < Bz; ++b) {
            for (int j = 0; j < ac; ++j) std::memcpy(&hA[b * nA + size_t(j) * ar], A + b * strideA + size_t(j) * lda, sizeof(double) * ar);
            for (int j = 0; j < N; ++j) std::memcpy(&hB[b * nB + size_t(j) * K], B + b * strideB + size_t(j) * ldb, sizeof(double) * K);
            for (int j = 0; j < N; ++j) std::memcpy(&hC[b * nC + size_t(j) * M], C + b * strideC + size_t(j) * ldc, sizeof(double) * M);
        }
        double *tA = nullptr, *tB = nullptr, *tC = nullptr;
        if ((rc = ws(h, "gemm_A", nA * Bz, &tA))) return rc;
        if ((rc = ws(h, "gemm_B", nB * Bz, &tB))) return rc;
        if ((rc = ws(h, "gemm_C", nC * Bz, &tC))) return rc;
        CU(cudaMemcpyAsync(tA, hA.data(), hA.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemcpyAsync(tB, hB.data(), hB.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemcpyAsync(tC, hC.data(), hC.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        LAUNCHED(dgemm_dmma_launch(transA, M, N, K, alpha, tA, ar, (long long)nA, tB, K, (long long)nB, beta, tC, M, (long long)nC, batch, h->stream));
        CU(cudaMemcpyAsync(hC.data(), tC, hC.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        for (size_t b = 0; b < Bz; ++b)
            for (int j = 0; j < N; ++j) std::memcpy(C + b * strideC + size_t(j) * ldc, &hC[b * nC + size_t(j) * M], sizeof(double) * M);
        return 0;
    }
    LAUNCHED(dgemm_dmma_launch(transA, M, N, K, alpha, dA, lda, sA, dB, ldb, sB, beta, dC, ldc, sC, batch, h->stream));
    return 0;
}

int copra_b200_lmpc_sizes(copra_b200_handle* h, const copra_b200_problem* p, copra_b200_sizes* s)
{
    if (!h || !s) return COPRA_B200_E_ARG;
    Plan pl;
    int rc = make_plan(h, p, pl);
    if (rc) return rc;
    s->X = pl.sz.X; s->nU = pl.sz.nU; s->nvar = pl.sz.nvar; s->meq = pl.sz.meq; s->mineq = pl.sz.mineq; s->q = pl.sz.q;
    return 0;
}

const char* copra_b200_last_solver(const copra_b200_handle* h) { return h ? h->solver : ""; }
int copra_b200_hessian_is_shared(const copra_b200_handle* h) { return (h && h->built && h->bp.sQ == 0) ? 1 : 0; }

int copra_b200_lmpc_built_sizes(copra_b200_handle* h, copra_b200_sizes* s)
{
    if (!h || !s) return COPRA_B200_E_ARG;
    if (!h->built) return fail(h, COPRA_B200_E_STATE, "no build is resident on this handle");
    s->X = h->sz.X; s->nU = h->sz.nU; s->nvar = h->sz.nvar; s->meq = h->sz.meq; s->mineq = h->sz.mineq; s->q = h->sz.q;
    return 0;
}

int copra_b200_lmpc_build(copra_b200_handle* h, const copra_b200_problem* p)
{
    if (!h) return COPRA_B200_E_ARG;
    h->built = false;
    return do_build(h, p);
}

int copra_b200_lmpc_solve(copra_b200_handle* h, const copra_b200_results* r)
{
    if (!h) return COPRA_B200_E_ARG;
    return do_solve(h, r);
}

int copra_b200_lmpc_run(copra_b200_handle* h, const copra_b200_problem* p, const copra_b200_results* r)
{
    if (!h) return COPRA_B200_E_ARG;
    h->built = false;
    h->qp_solved = false;
    if (!p) return fail(h, COPRA_B200_E_ARG, "null problem");
    const int kChunk = 32768;
    if (p->batch <= 65535) {
        int rc = do_build(h, p);
        if (rc) return rc;
        return do_solve(h, r);
    }
    // large batches: independent instances, so the batch is simply processed in chunks (the grid's y dimension
    // and the workspace stay bounded); every (pointer, stride) pair and every result pointer is advanced
    copra_b200_sizes sz;
    int rc = copra_b200_lmpc_sizes(h, p, &sz);
    if (rc) return rc;
    long long total_launches = 0;
    for (long long b0 = 0; b0 < p->batch; b0 += kChunk) {
        ProblemSlice q;
        slice_problem(*p, b0, int(std::min<long long>(kChunk, p->batch - b0)), q);
        copra_b200_results rr{};
        if (r) rr = slice_results(*r, b0, sz);
        if ((rc = do_build(h, &q.p))) return rc;
        if ((rc = do_solve(h, r ? &rr : nullptr))) return rc;
        total_launches += h->call_launches;
    }
    h->call_launches = total_launches;
    h->built = false; // the workspace only holds the last chunk
    return 0;
}

int copra_b200_fp64_peaks(copra_b200_handle* h, double* dfma_tflops, double* dmma_tflops)
{
    if (!h || !dfma_tflops || !dmma_tflops) return COPRA_B200_E_ARG;
    CU(cudaSetDevice(h->device));
    if (h->fp64_peaks[0] <= 0.0) {
        double* scratch = nullptr;
        int rc = ws(h, "peak_scratch", 1, &scratch);
        if (rc) return rc;
        const int r = fp64_peaks_measure(h->sms, scratch, h->stream, &h->fp64_peaks[0], &h->fp64_peaks[1]);
        if (r < 0) return fail(h, COPRA_B200_E_CUDA, "fp64_peaks: %s", cudaGetErrorString(cudaError_t(-r)));
        h->launches += 8;
    }
    *dfma_tflops = h->fp64_peaks[0];
    *dmma_tflops = h->fp64_peaks[1];
    return 0;
}

int copra_b200_lmpc_resolve(copra_b200_handle* h, copra_b200_array x0, int memory, const copra_b200_results* r)
{
    if (!h) return COPRA_B200_E_ARG;
    h->qp_solved = false;
    if (!h->built) return fail(h, COPRA_B200_E_STATE, "copra_b200_lmpc_resolve needs a previous build on this handle");
    BuildParams& P = h->bp;
    if (P.initial_state) return fail(h, COPRA_B200_E_UNSUPPORTED, "re-solve with new x0 is defined for LMPC mode only");
    if (!x0.ptr) return fail(h, COPRA_B200_E_ARG, "x0 is required");
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    for (bool& v : h->ev_valid) v = false;
    int rc = record(h, 0);
    if (rc) return rc;
    Upload U;
    U.add(x0, P.nx, &P.x0);
    if ((rc = run_upload(h, U, P.batch, memory, "params_x0"))) return rc; // its own buffer: the other parameters stay resident
    if ((rc = record(h, 1))) return rc;
    if ((rc = record(h, 2))) return rc;
    LAUNCHED(k4_finalize_launch(P, h->sms, h->stream));
    if ((rc = record(h, 3))) return rc;
    h->in_resolve = true;
    rc = do_solve(h, r);
    h->in_resolve = false;
    return rc;
}

int copra_b200_lmpc_retarget(copra_b200_handle* h, const copra_b200_problem* p, const copra_b200_results* r)
{
    if (!h) return COPRA_B200_E_ARG;
    h->qp_solved = false;
    if (!h->built) return fail(h, COPRA_B200_E_STATE, "copra_b200_lmpc_retarget needs a previous build on this handle");
    int rc = vector_inputs_check(h, "retarget");
    if (rc) return rc;
    BuildParams& P = h->bp;
    // everything is validated before BuildParams changes: a refused retarget leaves the resident build usable
    Plan pl;
    if ((rc = make_plan(h, p, pl, true))) return rc;
    if (shape_key(p, pl) != h->shape)
        return fail(h, COPRA_B200_E_ARG, "retarget: the problem's shape (dimensions, batch, entries, +-inf bound pattern) differs from the resident build");
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    for (bool& v : h->ev_valid) v = false;
    if ((rc = record(h, 0))) return rc;
    Upload U;
    BoundArrs ba;
    add_vectors(U, p, pl, P, ba);
    // its own buffer: the matrices stay resident in the build's
    if ((rc = run_upload(h, U, P.batch, p->memory, "params_vec"))) return rc;
    bind_bounds(pl, P, ba);
    if ((rc = record(h, 1))) return rc;
    if ((rc = record(h, 2))) return rc;
    LAUNCHED(k2_retarget_launch(P, h->sms, h->stream));
    LAUNCHED(k4_finalize_launch(P, h->sms, h->stream));
    if ((rc = record(h, 3))) return rc;
    h->in_resolve = true;
    rc = do_solve(h, r);
    h->in_resolve = false;
    return rc;
}

int copra_b200_lmpc_vjp(copra_b200_handle* h, const double* dcontrol, const double* dtrajectory, int memory,
    const copra_b200_vjp_out* out)
{
    return copra_b200_lmpc_vjp_costs(h, dcontrol, dtrajectory, memory, out, nullptr);
}

int copra_b200_lmpc_vjp_costs(copra_b200_handle* h, const double* dcontrol, const double* dtrajectory, int memory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_cost_out* costs)
{
    return copra_b200_lmpc_vjp_model(h, dcontrol, dtrajectory, memory, out, costs, nullptr);
}

int copra_b200_lmpc_vjp_model(copra_b200_handle* h, const double* dcontrol, const double* dtrajectory, int memory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_cost_out* costs, const copra_b200_vjp_model_out* model)
{
    if (!h) return COPRA_B200_E_ARG;
    if (!out && !costs && !model) return fail(h, COPRA_B200_E_ARG, "lmpc_vjp: null output description");
    if (memory != COPRA_B200_HOST && memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    int rc = sens_check(h, "lmpc_vjp");
    if (rc) return rc;
    if (costs) {
        const BuildParams& P = h->bp;
        for (int ci = 0; ci < P.ncost; ++ci) {
            if (costs->M && costs->M[ci] && !P.cost[ci].hasM)
                return fail(h, COPRA_B200_E_ARG, "lmpc_vjp_costs: cost %d has no M (a ControlCost)", ci);
            if (costs->N && costs->N[ci] && !P.cost[ci].hasN)
                return fail(h, COPRA_B200_E_ARG, "lmpc_vjp_costs: cost %d has no N (a TrajectoryCost or TargetCost)", ci);
        }
        if (k8_cost_grad_smem(P) > h->smem_optin)
            return fail(h, COPRA_B200_E_UNSUPPORTED, "lmpc_vjp_costs: the horizon needs %zu bytes of shared memory per instance, "
                "the device allows %zu", k8_cost_grad_smem(P), h->smem_optin);
    }
    if (model) {
        const BuildParams& P = h->bp;
        const int ncstr = int(h->cstr_len.size());
        std::vector<int> hasE(ncstr, 0), hasG(ncstr, 0);
        for (int fi = 0; fi < P.nfam; ++fi)
            if (h->fam_which[fi] == 0) {
                hasE[h->fam_cstr[fi]] = P.fam[fi].hasE;
                hasG[h->fam_cstr[fi]] = P.fam[fi].hasG;
            }
        for (int c = 0; c < ncstr; ++c) {
            if (model->E && model->E[c] && !hasE[c])
                return fail(h, COPRA_B200_E_ARG, "lmpc_vjp_model: constraint %d has no E (a ControlConstraint or a bound)", c);
            if (model->G && model->G[c] && !hasG[c])
                return fail(h, COPRA_B200_E_ARG, "lmpc_vjp_model: constraint %d has no G (a TrajectoryConstraint or a bound)", c);
        }
        if (k8_model_grad_smem(P) > h->smem_optin)
            return fail(h, COPRA_B200_E_UNSUPPORTED, "lmpc_vjp_model: the horizon needs %zu bytes of shared memory per instance, "
                "the device allows %zu", k8_model_grad_smem(P), h->smem_optin);
    }
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    return do_vjp(h, dcontrol, dtrajectory, memory, out, costs, model);
}

int copra_b200_lmpc_jvp(copra_b200_handle* h, const copra_b200_jvp_in* in, int memory, double* dcontrol, double* dtrajectory)
{
    if (!h) return COPRA_B200_E_ARG;
    if (!in) return fail(h, COPRA_B200_E_ARG, "lmpc_jvp: null tangent description");
    if (in->ndir < 1) return fail(h, COPRA_B200_E_ARG, "lmpc_jvp: ndir = %d, needs at least one direction", in->ndir);
    if (memory != COPRA_B200_HOST && memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    int rc = sens_check(h, "lmpc_jvp");
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    return do_jvp(h, in, in->ndir, false, memory, dcontrol, h->bp.nU, dtrajectory, h->bp.X);
}

int copra_b200_lmpc_feedback_gain(copra_b200_handle* h, int steps, double* Ku, double* Kx, int memory)
{
    if (!h) return COPRA_B200_E_ARG;
    if (memory != COPRA_B200_HOST && memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    int rc = sens_check(h, "lmpc_feedback_gain");
    if (rc) return rc;
    const BuildParams& P = h->bp;
    if (steps < 1 || steps > P.N) return fail(h, COPRA_B200_E_ARG, "lmpc_feedback_gain: steps = %d outside [1, N = %d]", steps, P.N);
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    return do_jvp(h, nullptr, P.nx, true, memory, Ku, P.nu * steps, Kx, P.nx * (steps + 1));
}

int copra_b200_lmpc_vjp_initial_state(copra_b200_handle* h, const double* dcontrol, const double* dtrajectory, int memory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_initial_out* init)
{
    if (!h) return COPRA_B200_E_ARG;
    if (memory != COPRA_B200_HOST && memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    static const copra_b200_vjp_initial_out none{};
    const copra_b200_vjp_initial_out& in = init ? *init : none;
    int rc = initial_state_check(h, "lmpc_vjp_initial_state", in.R, in.r, in.x0lb, in.x0ub, 1);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    return do_vjp(h, dcontrol, dtrajectory, memory, out, nullptr, nullptr, &in);
}

int copra_b200_lmpc_jvp_initial_state(copra_b200_handle* h, const copra_b200_jvp_in* in, const copra_b200_jvp_initial_in* init,
    int memory, double* dcontrol, double* dtrajectory)
{
    if (!h) return COPRA_B200_E_ARG;
    if (!in) return fail(h, COPRA_B200_E_ARG, "lmpc_jvp_initial_state: null tangent description");
    if (in->ndir < 1) return fail(h, COPRA_B200_E_ARG, "lmpc_jvp_initial_state: ndir = %d, needs at least one direction", in->ndir);
    if (memory != COPRA_B200_HOST && memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    static const copra_b200_jvp_initial_in none{};
    const copra_b200_jvp_initial_in& ti = init ? *init : none;
    int rc = initial_state_check(h, "lmpc_jvp_initial_state", ti.R, ti.r, ti.x0lb, ti.x0ub, in->ndir);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    return do_jvp(h, in, in->ndir, false, memory, dcontrol, h->bp.nU, dtrajectory, h->bp.X, &ti);
}

int copra_b200_set_warm_start(copra_b200_handle* h, int on)
{
    if (!h) return COPRA_B200_E_ARG;
    h->warm_start = on != 0;
    if (!on) h->warm_valid = false;
    return 0;
}

int copra_b200_get_warm_start(const copra_b200_handle* h) { return h && h->warm_start ? 1 : 0; }

int copra_b200_lmpc_results(copra_b200_handle* h, const double* x, double* control, double* trajectory, int memory)
{
    if (!h || !x) return COPRA_B200_E_ARG;
    if (!h->built) return fail(h, COPRA_B200_E_STATE, "results before build");
    const BuildParams& P = h->bp;
    const size_t B = P.batch;
    CU(cudaSetDevice(h->device));
    int rc;
    const double* dx = x;
    double *dc = control, *dt = trajectory;
    if (memory == COPRA_B200_HOST) {
        double* tmp = nullptr; // not res_x: that holds the solution of the last solve, for copra_b200_lmpc_vjp_costs
        if ((rc = ws(h, "results_x", B * P.nvar, &tmp))) return rc;
        CU(cudaMemcpyAsync(tmp, x, B * P.nvar * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        dx = tmp;
        if ((rc = ws(h, "res_control", B * P.nU, &dc))) return rc;
        if ((rc = ws(h, "res_traj", B * P.X, &dt))) return rc;
    }
    LAUNCHED(k7_results_launch(P, dx, control ? dc : nullptr, trajectory ? dt : nullptr, h->stream));
    if (memory == COPRA_B200_HOST) {
        if (control) CU(cudaMemcpyAsync(control, dc, B * P.nU * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (trajectory) CU(cudaMemcpyAsync(trajectory, dt, B * P.X * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

int copra_b200_lmpc_download(copra_b200_handle* h, int what, double* out, int memory)
{
    if (!h || !out) return COPRA_B200_E_ARG;
    if (!h->built) return fail(h, COPRA_B200_E_STATE, "download before build");
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    if (what == COPRA_B200_GET_AEQ || what == COPRA_B200_GET_AINEQ) {
        int rc = ensure_rows(h);
        if (rc) return rc;
    }
    const BuildParams& P = h->bp;
    const size_t B = P.batch, nv = P.nvar;
    const double* src = nullptr;
    size_t count = 0;
    // batch-invariant Hessian / per-cost E: one resident copy, replicated for the caller
    const bool oneE = what >= COPRA_B200_GET_COST_E && what < COPRA_B200_GET_COST_E + P.ncost && P.cost[what - COPRA_B200_GET_COST_E].sE == 0;
    if ((what == COPRA_B200_GET_Q && P.sQ == 0) || oneE) {
        const double* one = oneE ? P.cost[what - COPRA_B200_GET_COST_E].E : P.Q;
        const size_t cnt = oneE ? size_t(P.nx) * P.nU : nv * nv, bytes = cnt * sizeof(double);
        if (memory == COPRA_B200_DEVICE) {
            for (size_t b = 0; b < B; ++b) CU(cudaMemcpyAsync(out + b * cnt, one, bytes, cudaMemcpyDeviceToDevice, h->stream));
        } else {
            CU(cudaMemcpyAsync(out, one, bytes, cudaMemcpyDeviceToHost, h->stream));
            CU(cudaStreamSynchronize(h->stream));
            for (size_t b = 1; b < B; ++b) std::memcpy(out + b * cnt, out, bytes);
        }
        return 0;
    }
    switch (what) {
    case COPRA_B200_GET_PHI: src = P.Phi; count = B * P.X * P.nx; break;
    case COPRA_B200_GET_XI: src = P.xi; count = B * P.X; break;
    case COPRA_B200_GET_Q: src = P.Q; count = B * nv * nv; break;
    case COPRA_B200_GET_C: src = P.c; count = B * nv; break;
    case COPRA_B200_GET_AEQ: src = P.Aeq; count = B * P.meq * nv; break;
    case COPRA_B200_GET_BEQ: src = P.beq; count = B * P.meq; break;
    case COPRA_B200_GET_AINEQ: src = P.Aineq; count = B * P.mineq * nv; break;
    case COPRA_B200_GET_BINEQ: src = P.bineq; count = B * P.mineq; break;
    case COPRA_B200_GET_LB: src = P.lb; count = B * nv; break;
    case COPRA_B200_GET_UB: src = P.ub; count = B * nv; break;
    case COPRA_B200_GET_YEQ: src = P.Yeq; count = B * P.meq * P.nx; break;
    case COPRA_B200_GET_ZEQ: src = P.zeq; count = B * P.meq; break;
    case COPRA_B200_GET_YINEQ: src = P.Yin; count = B * P.mineq * P.nx; break;
    case COPRA_B200_GET_ZINEQ: src = P.zin; count = B * P.mineq; break;
    case COPRA_B200_GET_PSI: {
        count = B * size_t(P.X) * P.nU;
        double* psi = nullptr;
        if (memory == COPRA_B200_DEVICE) psi = out;
        else { int rc = ws(h, "Psi", count, &psi); if (rc) return rc; }
        LAUNCHED(k1_psi_fill_launch(P.Gs, (long long)P.N * P.nx * P.nu, psi, P.nx, P.nu, P.N, P.batch, h->stream));
        if (memory == COPRA_B200_DEVICE) return 0;
        src = psi;
    } break;
    default:
        if (what >= COPRA_B200_GET_COST_E && what < COPRA_B200_GET_COST_E + P.ncost) {
            src = P.cost[what - COPRA_B200_GET_COST_E].E; count = B * size_t(P.nx) * P.nU;
        } else if (what >= COPRA_B200_GET_COST_F && what < COPRA_B200_GET_COST_F + P.ncost) {
            src = P.cost[what - COPRA_B200_GET_COST_F].f; count = B * size_t(P.nU);
        } else return fail(h, COPRA_B200_E_ARG, "unknown download id %d", what);
    }
    if (count == 0) return 0;
    if (memory == COPRA_B200_DEVICE) CU(cudaMemcpyAsync(out, src, count * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    else {
        CU(cudaMemcpyAsync(out, src, count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

int copra_b200_condense(copra_b200_handle* h, int nx, int nu, int N, int batch, copra_b200_array A, copra_b200_array B,
    copra_b200_array d, double* Phi, double* Psi, double* xi, int memory)
{
    if (!h) return COPRA_B200_E_ARG;
    if (nx <= 0 || nu <= 0 || batch <= 0) return fail(h, COPRA_B200_E_ARG, "nx, nu and batch must be positive");
    if (N <= 0) return fail(h, COPRA_B200_E_ARG, "The number of step sould be a positive number!");
    if (!A.ptr || !B.ptr || !d.ptr) return fail(h, COPRA_B200_E_ARG, "A, B and d are required");
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    h->built = false;
    BuildParams P{};
    P.nx = nx; P.nu = nu; P.N = N; P.batch = batch; P.X = nx * (N + 1); P.nU = nu * N; P.nvar = P.nU;
    Upload U;
    U.add(A, size_t(nx) * nx, &P.A);
    U.add(B, size_t(nx) * nu, &P.B);
    U.add(d, nx, &P.d);
    int rc = run_upload(h, U, batch, memory, "params");
    if (rc) return rc;
    const size_t Bz = batch, X = P.X;
    const bool dv = memory == COPRA_B200_DEVICE;
    if (dv && Phi) P.Phi = Phi; else if ((rc = ws(h, "Phi", Bz * X * nx, &P.Phi))) return rc;
    if (dv && xi) P.xi = xi; else if ((rc = ws(h, "xi", Bz * X, &P.xi))) return rc;
    if ((rc = ws(h, "Gs", Bz * size_t(N) * nx * nu, &P.Gs))) return rc;
    LAUNCHED(k1_condense_launch(P, h->stream));
    double* psi = nullptr;
    if (Psi) {
        if (dv) psi = Psi; else if ((rc = ws(h, "Psi", Bz * X * P.nU, &psi))) return rc;
        LAUNCHED(k1_psi_fill_launch(P.Gs, (long long)N * nx * nu, psi, nx, nu, N, batch, h->stream));
    }
    if (!dv) {
        if (Phi) CU(cudaMemcpyAsync(Phi, P.Phi, Bz * X * nx * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (xi) CU(cudaMemcpyAsync(xi, P.xi, Bz * X * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (Psi) CU(cudaMemcpyAsync(Psi, psi, Bz * X * P.nU * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

int copra_b200_solve_qp_batch(copra_b200_handle* h, int n, int meq, int m, int batch, copra_b200_array Q, copra_b200_array c,
    copra_b200_array Aeq, copra_b200_array beq, copra_b200_array Aineq, copra_b200_array bineq, copra_b200_array lb,
    copra_b200_array ub, double* x, int* status, int* iters, int* nact, int* iact, int memory)
{
    if (!h) return COPRA_B200_E_ARG;
    if (n <= 0 || meq < 0 || m < 0 || batch <= 0) return fail(h, COPRA_B200_E_ARG, "bad QP dimensions");
    if (!Q.ptr || !c.ptr || !lb.ptr || !ub.ptr) return fail(h, COPRA_B200_E_ARG, "Q, c, lb and ub are required");
    if ((meq > 0 && (!Aeq.ptr || !beq.ptr)) || (m > 0 && (!Aineq.ptr || !bineq.ptr))) return fail(h, COPRA_B200_E_ARG, "constraint matrices missing");
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    /* the last lmpc build stays valid: this entry uses its own workspace buffers, except for the active sets */
    h->solved = false;
    h->qp_solved = false;
    for (bool& v : h->ev_valid) v = false;
    int rc = record(h, 0);
    if (rc) return rc;
    GiBatch G{};
    G.n = n; G.meq = meq; G.m = m; G.batch = batch;
    Upload U;
    U.add(Q, size_t(n) * n, &G.Q);
    U.add(c, n, &G.c);
    if (meq) { U.add(Aeq, size_t(meq) * n, &G.Aeq); U.add(beq, meq, &G.beq); }
    if (m) { U.add(Aineq, size_t(m) * n, &G.Aineq); U.add(bineq, m, &G.bineq); }
    U.add(lb, n, &G.lb);
    U.add(ub, n, &G.ub);
    if ((rc = run_upload(h, U, batch, memory, "qp_params"))) return rc;
    if ((rc = record(h, 1))) return rc;
    h->ev_valid[2] = h->ev_valid[3] = false;
    const size_t B = batch;
    const bool dv = memory == COPRA_B200_DEVICE;
    if (dv && x) G.x = x; else if ((rc = ws(h, "res_x", B * n, &G.x))) return rc;
    if (dv && status) G.status = status; else if ((rc = ws(h, "res_status", B, &G.status))) return rc;
    if (dv && iters) G.iters = iters; else if ((rc = ws(h, "res_iters", 2 * B, &G.iters))) return rc;
    if (dv && nact) G.nact = nact; else if ((rc = ws(h, "res_nact", B, &G.nact))) return rc;
    if (dv && iact) G.iact = iact; else if ((rc = ws(h, "res_iact", B * n, &G.iact))) return rc;
    if ((rc = record(h, 3))) return rc;
    if ((rc = run_gi(h, G))) return rc;
    if ((rc = record(h, 4))) return rc;
    // the solution and the active sets stay in the workspace for copra_b200_qp_vjp
    const auto keep = [&](const char* name, void* src, size_t bytes) {
        void* dst = nullptr;
        int rc2 = dev_reserve(h, name, bytes, &dst);
        if (rc2 || dst == src) return rc2;
        CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, h->stream));
        return 0;
    };
    if ((rc = keep("res_x", G.x, B * n * sizeof(double)))) return rc;
    if ((rc = keep("res_status", G.status, B * sizeof(int)))) return rc;
    if ((rc = keep("res_nact", G.nact, B * sizeof(int)))) return rc;
    if ((rc = keep("res_iact", G.iact, B * n * sizeof(int)))) return rc;
    if ((rc = record(h, 5))) return rc;
    if (!dv) {
        Download D;
        D.add(G.x, x, B * n * sizeof(double));
        D.add(G.status, status, B * sizeof(int));
        D.add(G.iters, iters, 2 * B * sizeof(int));
        D.add(G.nact, nact, B * sizeof(int));
        D.add(G.iact, iact, B * n * sizeof(int));
        if ((rc = run_download(h, D, COPRA_B200_HOST))) return rc;
    }
    if ((rc = record(h, 6))) return rc;
    h->qp = G;
    h->qp_solved = true;
    return 0;
}

int copra_b200_qp_vjp(copra_b200_handle* h, const double* dx, int memory, const copra_b200_qp_vjp_out* out)
{
    if (!h) return COPRA_B200_E_ARG;
    if (!h->qp_solved)
        return fail(h, COPRA_B200_E_STATE, "copra_b200_qp_vjp needs a raw QP batch (copra_b200_solve_qp_batch) as the last solve on this handle");
    if (!dx) return fail(h, COPRA_B200_E_ARG, "qp_vjp: dx is required");
    if (memory != COPRA_B200_HOST && memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    const GiBatch& G = h->qp;
    if (!out) return 0;
    if ((out->Aeq || out->beq) && G.meq == 0) return fail(h, COPRA_B200_E_ARG, "qp_vjp: dAeq / dbeq requested for a batch without equality rows");
    if ((out->Aineq || out->bineq) && G.m == 0) return fail(h, COPRA_B200_E_ARG, "qp_vjp: dAineq / dbineq requested for a batch without inequality rows");
    const int k = (out->Aeq || out->Aineq) ? 2 : 1;
    // qp_grad holds v and x, sens_solve up to 2 k n doubles (the active set has at most n rows), gt_factor Q's scratch
    const size_t smem = std::max(std::max(qp_grad_smem(G.n), sizeof(double) * 2 * k * size_t(G.n)), gt_factor_smem(G.n));
    if (smem > h->smem_optin)
        return fail(h, COPRA_B200_E_UNSUPPORTED, "qp_vjp: n = %d needs %zu bytes of shared memory per block, the device allows %zu",
            G.n, smem, h->smem_optin);
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    return do_qp_vjp(h, dx, memory, out);
}

// the shared preconditions of copra_b200_qp_jvp / copra_b200_qp_jacobian with k directions: sens_solve's shared memory for k
// right-hand sides (the active set has at most n rows) and gt_factor's for Q within the device's limit
static int qp_jvp_check(copra_b200_handle* h, const char* name, int k)
{
    const GiBatch& G = h->qp;
    const size_t smem = std::max(sens_solve_smem(k, G.n), gt_factor_smem(G.n));
    if (smem > h->smem_optin)
        return fail(h, COPRA_B200_E_UNSUPPORTED, "%s: n = %d needs %zu bytes of shared memory per block, the device allows %zu",
            name, G.n, smem, h->smem_optin);
    return 0;
}

int copra_b200_qp_jvp(copra_b200_handle* h, const copra_b200_qp_jvp_in* in, int memory, double* dx)
{
    if (!h) return COPRA_B200_E_ARG;
    if (!h->qp_solved)
        return fail(h, COPRA_B200_E_STATE, "copra_b200_qp_jvp needs a raw QP batch (copra_b200_solve_qp_batch) as the last solve on this handle");
    if (!in) return fail(h, COPRA_B200_E_ARG, "qp_jvp: the tangents are required");
    if (memory != COPRA_B200_HOST && memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    if (in->ndir < 1) return fail(h, COPRA_B200_E_ARG, "qp_jvp: ndir = %d, needs at least one direction", in->ndir);
    const copra_b200_array* t[] = { &in->Q, &in->c, &in->Aeq, &in->beq, &in->Aineq, &in->bineq, &in->lb, &in->ub };
    for (const copra_b200_array* a : t)
        if (a->ptr && a->stride < 0) return fail(h, COPRA_B200_E_ARG, "qp_jvp: negative tangent stride %lld", a->stride);
    const GiBatch& G = h->qp;
    if ((in->Aeq.ptr || in->beq.ptr) && G.meq == 0) return fail(h, COPRA_B200_E_ARG, "qp_jvp: Aeq / beq tangents for a batch without equality rows");
    if ((in->Aineq.ptr || in->bineq.ptr) && G.m == 0) return fail(h, COPRA_B200_E_ARG, "qp_jvp: Aineq / bineq tangents for a batch without inequality rows");
    int rc = qp_jvp_check(h, "qp_jvp", in->ndir);
    if (rc || !dx) return rc;
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    return do_qp_jvp(h, in, in->ndir, -1, memory, dx);
}

int copra_b200_qp_jacobian(copra_b200_handle* h, int wrt, double* J, int memory)
{
    if (!h) return COPRA_B200_E_ARG;
    if (!h->qp_solved)
        return fail(h, COPRA_B200_E_STATE, "copra_b200_qp_jacobian needs a raw QP batch (copra_b200_solve_qp_batch) as the last solve on this handle");
    if (memory != COPRA_B200_HOST && memory != COPRA_B200_DEVICE) return fail(h, COPRA_B200_E_ARG, "bad memory kind");
    const GiBatch& G = h->qp;
    int len;
    switch (wrt) {
    case COPRA_B200_QP_WRT_C: len = G.n; break;
    case COPRA_B200_QP_WRT_BEQ: len = G.meq; break;
    case COPRA_B200_QP_WRT_BINEQ: len = G.m; break;
    case COPRA_B200_QP_WRT_LB: case COPRA_B200_QP_WRT_UB: len = G.n; break;
    default: return fail(h, COPRA_B200_E_ARG, "qp_jacobian: unknown wrt %d", wrt);
    }
    if (len == 0) return fail(h, COPRA_B200_E_ARG, "qp_jacobian: wrt %d names rows the batch does not have", wrt);
    int rc = qp_jvp_check(h, "qp_jacobian", len);
    if (rc || !J) return rc;
    CU(cudaSetDevice(h->device));
    h->call_launches = 0;
    return do_qp_jvp(h, nullptr, len, wrt, memory, J);
}

} // extern "C"
