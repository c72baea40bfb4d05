// capi_multi.cu -- the data-parallel sharder of the batched engine (SURVEY.md 8e): a batch of independent controllers is
// split by instance index into contiguous ranges [g*ceil(B/G), (g+1)*ceil(B/G)), one range per device.  Every device has
// its own engine handle (stream, workspace, pinned staging) driven by its own host thread; parameters go up per shard
// and the results of every shard are written by DMA straight into the caller's (ideally page-locked) result buffers --
// that final gather is the only cross-device step, there is no collective on the path.  Built on the public
// single-device C ABI only, so the results of a shard are bit-identical to a single-device run of the same instances.
#include "../../include/copra_b200.h"
#include "slice.h"

#include <algorithm>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

using namespace cb;

struct copra_b200_multi {
    std::vector<copra_b200_handle*> h;
    std::vector<int> dev;
    std::vector<int> lo, hi;   // shard ranges of the last run
    std::vector<int> rc;
    std::string err;
    double wall_ms = 0.0;
};

namespace {

int mfail(copra_b200_multi* m, int code, const std::string& msg)
{
    if (m) m->err = msg;
    return code;
}

void shard_ranges(copra_b200_multi* m, int batch)
{
    const int G = int(m->h.size());
    const int per = (batch + G - 1) / G;
    m->lo.assign(G, 0);
    m->hi.assign(G, 0);
    for (int g = 0; g < G; ++g) {
        m->lo[g] = std::min(batch, g * per);
        m->hi[g] = std::min(batch, (g + 1) * per);
    }
}

template <class F> int run_shards(copra_b200_multi* m, F body)
{
    const int G = int(m->h.size());
    m->rc.assign(G, 0);
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::thread> th;
    for (int g = 1; g < G; ++g)
        if (m->hi[g] > m->lo[g]) th.emplace_back([&, g] { m->rc[g] = body(g); });
    if (m->hi[0] > m->lo[0]) m->rc[0] = body(0); // the calling thread drives device 0's shard
    for (auto& t : th) t.join();
    m->wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    for (int g = 0; g < G; ++g)
        if (m->rc[g]) return mfail(m, m->rc[g], "device " + std::to_string(m->dev[g]) + ": " + copra_b200_last_error(m->h[g]));
    return 0;
}

} // namespace

// per-instance lengths of x0 and of every cost's p / constraint's vector of the resident build (capi.cu)
void cb_vjp_lengths(const copra_b200_handle* h, int& nx, std::vector<int>& cost_len, std::vector<int>& cstr_len);
// nu and the rows of every cost of the resident build (capi.cu)
void cb_cost_shapes(const copra_b200_handle* h, int& nu, std::vector<int>& rows);
// the rows of every row constraint's E / G of the resident build, 0 for a bound (capi.cu)
void cb_cstr_rows(const copra_b200_handle* h, std::vector<int>& rows);

namespace {

// the per-instance shapes of a shard's resident build: nx, nu, the lengths of every cost's p and every constraint's
// vector, the rows of every cost and of every row constraint's E / G (0 for a bound)
struct ShardShapes {
    int nx = 0, nu = 0;
    std::vector<int> plen, clen, cost_rows, cstr_rows;
    explicit ShardShapes(const copra_b200_handle* h)
    {
        cb_vjp_lengths(h, nx, plen, clen);
        cb_cost_shapes(h, nu, cost_rows);
        cb_cstr_rows(h, cstr_rows);
    }
};

// arr[i] + lo * len[i] * k for every entry i of a whole-batch pointer array (null stays null)
template <class T> std::vector<T*> advance(T* const* arr, const std::vector<int>& len, long long lo, long long k = 1)
{
    std::vector<T*> out(len.size());
    for (size_t i = 0; i < len.size(); ++i) out[i] = (arr && arr[i]) ? arr[i] + lo * len[i] * k : nullptr;
    return out;
}

// Runs a VJP over the shards: the whole-batch cotangents and outputs (vectors; cost, model and initial-state gradients
// where asked for) are advanced to each shard's first instance and handed to copra_b200_lmpc_vjp_initial_state when
// `initial`, to copra_b200_lmpc_vjp_model otherwise.  `name` is the entry's name in the error strings.
int multi_vjp(copra_b200_multi* m, const char* name, bool initial, const double* dcontrol, const double* dtrajectory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_cost_out* costs, const copra_b200_vjp_model_out* model,
    const copra_b200_vjp_initial_out* init)
{
    if (!m) return COPRA_B200_E_ARG;
    if (!initial && !out && !costs && !model) return mfail(m, COPRA_B200_E_ARG, std::string(name) + ": null output description");
    static const copra_b200_vjp_out none{};
    if (!out) out = &none;
    if (m->lo.size() != m->h.size()) return mfail(m, COPRA_B200_E_STATE, std::string("copra_b200_multi_") + name + " needs a previous run");
    return run_shards(m, [&](int g) {
        copra_b200_sizes sz{};
        int rc = copra_b200_lmpc_built_sizes(m->h[g], &sz);
        if (rc) return rc;
        const ShardShapes s(m->h[g]);
        const int nx = s.nx, nu = s.nu;
        const long long lo = m->lo[g];
        std::vector<double*> p = advance(out->p, s.plen, lo), f = advance(out->f, s.clen, lo),
                             lower = advance(out->lower, s.clen, lo), upper = advance(out->upper, s.clen, lo);
        copra_b200_vjp_out o{};
        o.x0 = out->x0 ? out->x0 + lo * nx : nullptr;
        o.p = out->p ? p.data() : nullptr;
        o.f = out->f ? f.data() : nullptr;
        o.lower = out->lower ? lower.data() : nullptr;
        o.upper = out->upper ? upper.data() : nullptr;
        // the cost gradients: rows, rows x nx and rows x nu per instance
        std::vector<double*> cw, cM, cN;
        copra_b200_vjp_cost_out co{};
        if (costs) {
            cw = advance(costs->w, s.cost_rows, lo), cM = advance(costs->M, s.cost_rows, lo, nx);
            cN = advance(costs->N, s.cost_rows, lo, nu);
            co.w = costs->w ? cw.data() : nullptr;
            co.M = costs->M ? cM.data() : nullptr;
            co.N = costs->N ? cN.data() : nullptr;
        }
        // the model gradients: nx x nx, nx x nu, nx, and rows x nx / rows x nu per row constraint
        std::vector<double*> mE, mG;
        copra_b200_vjp_model_out mo{};
        if (model) {
            mE = advance(model->E, s.cstr_rows, lo, nx), mG = advance(model->G, s.cstr_rows, lo, nu);
            mo.A = model->A ? model->A + lo * nx * nx : nullptr;
            mo.B = model->B ? model->B + lo * nx * nu : nullptr;
            mo.d = model->d ? model->d + lo * nx : nullptr;
            mo.E = model->E ? mE.data() : nullptr;
            mo.G = model->G ? mG.data() : nullptr;
        }
        // the initial-state gradients: nx x nx, nx, nx, nx
        copra_b200_vjp_initial_out io{};
        if (init) {
            io.R = init->R ? init->R + lo * nx * nx : nullptr;
            io.r = init->r ? init->r + lo * nx : nullptr;
            io.x0lb = init->x0lb ? init->x0lb + lo * nx : nullptr;
            io.x0ub = init->x0ub ? init->x0ub + lo * nx : nullptr;
        }
        const double* dc = dcontrol ? dcontrol + lo * sz.nU : nullptr;
        const double* dt = dtrajectory ? dtrajectory + lo * sz.X : nullptr;
        if (initial) return copra_b200_lmpc_vjp_initial_state(m->h[g], dc, dt, COPRA_B200_HOST, &o, init ? &io : nullptr);
        return copra_b200_lmpc_vjp_model(m->h[g], dc, dt, COPRA_B200_HOST, &o, costs ? &co : nullptr, model ? &mo : nullptr);
    });
}

// Runs a JVP over the shards: the whole-batch tangents (len x k per instance: vectors, and R, r, x0lb, x0ub where given)
// and outputs are advanced to each shard's first instance and handed to copra_b200_lmpc_jvp_initial_state when
// `initial`, to copra_b200_lmpc_jvp otherwise.  `name` is the entry's name in the error strings.
int multi_jvp(copra_b200_multi* m, const char* name, bool initial, const copra_b200_jvp_in* in,
    const copra_b200_jvp_initial_in* init, double* dcontrol, double* dtrajectory)
{
    if (!m) return COPRA_B200_E_ARG;
    if (!in) return mfail(m, COPRA_B200_E_ARG, std::string(name) + ": null tangent description");
    if (m->lo.size() != m->h.size()) return mfail(m, COPRA_B200_E_STATE, std::string("copra_b200_multi_") + name + " needs a previous run");
    return run_shards(m, [&](int g) {
        copra_b200_sizes sz{};
        int rc = copra_b200_lmpc_built_sizes(m->h[g], &sz);
        if (rc) return rc;
        const ShardShapes s(m->h[g]);
        const long long nx = s.nx, lo = m->lo[g], k = in->ndir;
        std::vector<const double*> p = advance(in->p, s.plen, lo, k), f = advance(in->f, s.clen, lo, k),
                                   lower = advance(in->lower, s.clen, lo, k), upper = advance(in->upper, s.clen, lo, k);
        copra_b200_jvp_in t = *in;
        t.x0 = in->x0 ? in->x0 + lo * nx * k : nullptr;
        t.p = in->p ? p.data() : nullptr;
        t.f = in->f ? f.data() : nullptr;
        t.lower = in->lower ? lower.data() : nullptr;
        t.upper = in->upper ? upper.data() : nullptr;
        copra_b200_jvp_initial_in ti{};
        if (init) {
            ti.R = init->R ? init->R + lo * nx * nx * k : nullptr;
            ti.r = init->r ? init->r + lo * nx * k : nullptr;
            ti.x0lb = init->x0lb ? init->x0lb + lo * nx * k : nullptr;
            ti.x0ub = init->x0ub ? init->x0ub + lo * nx * k : nullptr;
        }
        double* du = dcontrol ? dcontrol + lo * sz.nU * k : nullptr;
        double* dx = dtrajectory ? dtrajectory + lo * sz.X * k : nullptr;
        if (initial) return copra_b200_lmpc_jvp_initial_state(m->h[g], &t, init ? &ti : nullptr, COPRA_B200_HOST, du, dx);
        return copra_b200_lmpc_jvp(m->h[g], &t, COPRA_B200_HOST, du, dx);
    });
}

} // namespace

extern "C" {

int copra_b200_multi_create(const int* devices, int ndev, copra_b200_multi** out)
{
    if (!out) return COPRA_B200_E_ARG;
    *out = nullptr;
    const int avail = copra_b200_device_count();
    if (avail <= 0) return COPRA_B200_E_NOGPU;
    std::vector<int> devs;
    if (!devices || ndev <= 0) for (int d = 0; d < avail; ++d) devs.push_back(d);
    else devs.assign(devices, devices + ndev);
    copra_b200_multi* m = new copra_b200_multi();
    for (int d : devs) {
        copra_b200_options opt{};
        opt.device = d;
        copra_b200_handle* h = nullptr;
        const int rc = copra_b200_create(&opt, &h);
        if (rc) {
            for (auto* hh : m->h) copra_b200_destroy(hh);
            delete m;
            return rc;
        }
        m->h.push_back(h);
        m->dev.push_back(d);
    }
    *out = m;
    return COPRA_B200_OK;
}

void copra_b200_multi_destroy(copra_b200_multi* m)
{
    if (!m) return;
    for (auto* h : m->h) copra_b200_destroy(h);
    delete m;
}

const char* copra_b200_multi_last_error(const copra_b200_multi* m) { return m ? m->err.c_str() : "null handle"; }
int copra_b200_multi_size(const copra_b200_multi* m) { return m ? int(m->h.size()) : 0; }

int copra_b200_multi_shard(const copra_b200_multi* m, int g, int* device, int* lo, int* hi)
{
    if (!m || g < 0 || g >= int(m->h.size())) return COPRA_B200_E_ARG;
    if (device) *device = m->dev[g];
    if (lo) *lo = g < int(m->lo.size()) ? m->lo[g] : 0;
    if (hi) *hi = g < int(m->hi.size()) ? m->hi[g] : 0;
    return 0;
}

int copra_b200_multi_timing(const copra_b200_multi* m, int g, copra_b200_timing* t, double* wall_ms)
{
    if (!m || g < 0 || g >= int(m->h.size())) return COPRA_B200_E_ARG;
    if (wall_ms) *wall_ms = m->wall_ms;
    return t ? copra_b200_last_timing(m->h[g], t) : 0;
}

long long copra_b200_multi_launch_count(const copra_b200_multi* m)
{
    long long n = 0;
    if (m) for (auto* h : m->h) n += copra_b200_launch_count(h);
    return n;
}

int copra_b200_multi_lmpc_run(copra_b200_multi* m, const copra_b200_problem* p, const copra_b200_results* r)
{
    if (!m) return COPRA_B200_E_ARG;
    if (!p) return mfail(m, COPRA_B200_E_ARG, "null problem");
    if (p->memory != COPRA_B200_HOST || (r && r->memory != COPRA_B200_HOST))
        return mfail(m, COPRA_B200_E_ARG, "the multi-device entry takes HOST arrays (each shard is uploaded to its own device)");
    copra_b200_sizes sz;
    int rc = copra_b200_lmpc_sizes(m->h[0], p, &sz);
    if (rc) return mfail(m, rc, copra_b200_last_error(m->h[0]));
    shard_ranges(m, p->batch);
    return run_shards(m, [&](int g) {
        ProblemSlice q;
        slice_problem(*p, m->lo[g], m->hi[g] - m->lo[g], q);
        copra_b200_results rr{};
        if (r) rr = slice_results(*r, m->lo[g], sz);
        return copra_b200_lmpc_run(m->h[g], &q.p, r ? &rr : nullptr);
    });
}

int copra_b200_multi_set_warm_start(copra_b200_multi* m, int on)
{
    if (!m) return COPRA_B200_E_ARG;
    for (copra_b200_handle* h : m->h) copra_b200_set_warm_start(h, on);
    return 0;
}

int copra_b200_multi_lmpc_resolve(copra_b200_multi* m, copra_b200_array x0, const copra_b200_results* r)
{
    if (!m) return COPRA_B200_E_ARG;
    if (!x0.ptr) return mfail(m, COPRA_B200_E_ARG, "x0 is required");
    if (m->lo.size() != m->h.size()) return mfail(m, COPRA_B200_E_STATE, "copra_b200_multi_lmpc_resolve needs a previous run");
    if (r && r->memory != COPRA_B200_HOST) return mfail(m, COPRA_B200_E_ARG, "the multi-device entry takes HOST arrays");
    return run_shards(m, [&](int g) {
        copra_b200_results rr{};
        if (r) {
            // per-instance result sizes are those of the resident build: recover them from the shard's own handle
            copra_b200_sizes sz{};
            const int rc = copra_b200_lmpc_built_sizes(m->h[g], &sz);
            if (rc) return rc;
            rr = slice_results(*r, m->lo[g], sz);
        }
        return copra_b200_lmpc_resolve(m->h[g], slice_array(x0, m->lo[g]), COPRA_B200_HOST, r ? &rr : nullptr);
    });
}

int copra_b200_multi_lmpc_retarget(copra_b200_multi* m, const copra_b200_problem* p, const copra_b200_results* r)
{
    if (!m) return COPRA_B200_E_ARG;
    if (!p) return mfail(m, COPRA_B200_E_ARG, "null problem");
    if (p->memory != COPRA_B200_HOST || (r && r->memory != COPRA_B200_HOST))
        return mfail(m, COPRA_B200_E_ARG, "the multi-device entry takes HOST arrays (each shard is uploaded to its own device)");
    if (m->lo.size() != m->h.size()) return mfail(m, COPRA_B200_E_STATE, "copra_b200_multi_lmpc_retarget needs a previous run");
    if (p->batch != m->hi.back()) return mfail(m, COPRA_B200_E_ARG, "retarget: the batch differs from the resident run's");
    return run_shards(m, [&](int g) {
        ProblemSlice q;
        slice_problem(*p, m->lo[g], m->hi[g] - m->lo[g], q);
        copra_b200_results rr{};
        if (r) {
            copra_b200_sizes sz{};
            const int rc = copra_b200_lmpc_built_sizes(m->h[g], &sz);
            if (rc) return rc;
            rr = slice_results(*r, m->lo[g], sz);
        }
        return copra_b200_lmpc_retarget(m->h[g], &q.p, r ? &rr : nullptr);
    });
}

int copra_b200_multi_lmpc_vjp(copra_b200_multi* m, const double* dcontrol, const double* dtrajectory, const copra_b200_vjp_out* out)
{
    return copra_b200_multi_lmpc_vjp_costs(m, dcontrol, dtrajectory, out, nullptr);
}

int copra_b200_multi_lmpc_vjp_costs(copra_b200_multi* m, const double* dcontrol, const double* dtrajectory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_cost_out* costs)
{
    return copra_b200_multi_lmpc_vjp_model(m, dcontrol, dtrajectory, out, costs, nullptr);
}

int copra_b200_multi_lmpc_vjp_model(copra_b200_multi* m, const double* dcontrol, const double* dtrajectory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_cost_out* costs, const copra_b200_vjp_model_out* model)
{
    return multi_vjp(m, "lmpc_vjp", false, dcontrol, dtrajectory, out, costs, model, nullptr);
}

int copra_b200_multi_lmpc_jvp(copra_b200_multi* m, const copra_b200_jvp_in* in, double* dcontrol, double* dtrajectory)
{
    return multi_jvp(m, "lmpc_jvp", false, in, nullptr, dcontrol, dtrajectory);
}

int copra_b200_multi_lmpc_vjp_initial_state(copra_b200_multi* m, const double* dcontrol, const double* dtrajectory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_initial_out* init)
{
    return multi_vjp(m, "lmpc_vjp_initial_state", true, dcontrol, dtrajectory, out, nullptr, nullptr, init);
}

int copra_b200_multi_lmpc_jvp_initial_state(copra_b200_multi* m, const copra_b200_jvp_in* in, const copra_b200_jvp_initial_in* init,
    double* dcontrol, double* dtrajectory)
{
    return multi_jvp(m, "lmpc_jvp_initial_state", true, in, init, dcontrol, dtrajectory);
}

int copra_b200_multi_lmpc_feedback_gain(copra_b200_multi* m, int steps, double* Ku, double* Kx)
{
    if (!m) return COPRA_B200_E_ARG;
    if (m->lo.size() != m->h.size()) return mfail(m, COPRA_B200_E_STATE, "copra_b200_multi_lmpc_feedback_gain needs a previous run");
    return run_shards(m, [&](int g) {
        copra_b200_sizes sz{};
        int rc = copra_b200_lmpc_built_sizes(m->h[g], &sz);
        if (rc) return rc;
        const int nx = ShardShapes(m->h[g]).nx;
        const int N = sz.X / nx - 1, nu = N > 0 ? sz.nU / N : 0;
        if (steps < 1 || steps > N) return copra_b200_lmpc_feedback_gain(m->h[g], steps, nullptr, nullptr, COPRA_B200_HOST); // E_ARG
        const long long lo = m->lo[g];
        return copra_b200_lmpc_feedback_gain(m->h[g], steps, Ku ? Ku + lo * nu * steps * nx : nullptr,
            Kx ? Kx + lo * nx * (steps + 1) * nx : nullptr, COPRA_B200_HOST);
    });
}

} // extern "C"
