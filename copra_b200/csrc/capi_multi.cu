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
    if (!m) return COPRA_B200_E_ARG;
    if (!out && !costs && !model) return mfail(m, COPRA_B200_E_ARG, "lmpc_vjp: null output description");
    static const copra_b200_vjp_out none{};
    if (!out) out = &none;
    if (m->lo.size() != m->h.size()) return mfail(m, COPRA_B200_E_STATE, "copra_b200_multi_lmpc_vjp needs a previous run");
    return run_shards(m, [&](int g) {
        copra_b200_sizes sz{};
        int rc = copra_b200_lmpc_built_sizes(m->h[g], &sz);
        if (rc) return rc;
        std::vector<int> plen, clen;
        int nx = 0;
        cb_vjp_lengths(m->h[g], nx, plen, clen);
        const long long lo = m->lo[g];
        // every array of the whole batch, advanced to this shard's first instance
        std::vector<double*> p(plen.size()), f(clen.size()), lower(clen.size()), upper(clen.size());
        for (size_t i = 0; i < plen.size(); ++i) p[i] = (out->p && out->p[i]) ? out->p[i] + lo * plen[i] : nullptr;
        for (size_t i = 0; i < clen.size(); ++i) {
            f[i] = (out->f && out->f[i]) ? out->f[i] + lo * clen[i] : nullptr;
            lower[i] = (out->lower && out->lower[i]) ? out->lower[i] + lo * clen[i] : nullptr;
            upper[i] = (out->upper && out->upper[i]) ? out->upper[i] + lo * clen[i] : nullptr;
        }
        copra_b200_vjp_out o{};
        o.x0 = out->x0 ? out->x0 + lo * nx : nullptr;
        o.p = out->p ? p.data() : nullptr;
        o.f = out->f ? f.data() : nullptr;
        o.lower = out->lower ? lower.data() : nullptr;
        o.upper = out->upper ? upper.data() : nullptr;
        // the cost gradients likewise: rows, rows x nx and rows x nu per instance
        int nu = 0;
        std::vector<int> rows;
        cb_cost_shapes(m->h[g], nu, rows);
        std::vector<double*> cw(rows.size()), cM(rows.size()), cN(rows.size());
        for (size_t i = 0; i < rows.size() && costs; ++i) {
            cw[i] = (costs->w && costs->w[i]) ? costs->w[i] + lo * rows[i] : nullptr;
            cM[i] = (costs->M && costs->M[i]) ? costs->M[i] + lo * rows[i] * nx : nullptr;
            cN[i] = (costs->N && costs->N[i]) ? costs->N[i] + lo * rows[i] * nu : nullptr;
        }
        copra_b200_vjp_cost_out co{};
        if (costs) {
            co.w = costs->w ? cw.data() : nullptr;
            co.M = costs->M ? cM.data() : nullptr;
            co.N = costs->N ? cN.data() : nullptr;
        }
        // and the model gradients: nx x nx, nx x nu, nx, and rows x nx / rows x nu per row constraint
        std::vector<int> crows;
        cb_cstr_rows(m->h[g], crows);
        std::vector<double*> mE(crows.size()), mG(crows.size());
        for (size_t i = 0; i < crows.size() && model; ++i) {
            mE[i] = (model->E && model->E[i]) ? model->E[i] + lo * crows[i] * nx : nullptr;
            mG[i] = (model->G && model->G[i]) ? model->G[i] + lo * crows[i] * nu : nullptr;
        }
        copra_b200_vjp_model_out mo{};
        if (model) {
            mo.A = model->A ? model->A + lo * nx * nx : nullptr;
            mo.B = model->B ? model->B + lo * nx * nu : nullptr;
            mo.d = model->d ? model->d + lo * nx : nullptr;
            mo.E = model->E ? mE.data() : nullptr;
            mo.G = model->G ? mG.data() : nullptr;
        }
        return copra_b200_lmpc_vjp_model(m->h[g], dcontrol ? dcontrol + lo * sz.nU : nullptr,
            dtrajectory ? dtrajectory + lo * sz.X : nullptr, COPRA_B200_HOST, &o, costs ? &co : nullptr, model ? &mo : nullptr);
    });
}

int copra_b200_multi_lmpc_jvp(copra_b200_multi* m, const copra_b200_jvp_in* in, double* dcontrol, double* dtrajectory)
{
    if (!m) return COPRA_B200_E_ARG;
    if (!in) return mfail(m, COPRA_B200_E_ARG, "lmpc_jvp: null tangent description");
    if (m->lo.size() != m->h.size()) return mfail(m, COPRA_B200_E_STATE, "copra_b200_multi_lmpc_jvp needs a previous run");
    return run_shards(m, [&](int g) {
        copra_b200_sizes sz{};
        int rc = copra_b200_lmpc_built_sizes(m->h[g], &sz);
        if (rc) return rc;
        std::vector<int> plen, clen;
        int nx = 0;
        cb_vjp_lengths(m->h[g], nx, plen, clen);
        const long long lo = m->lo[g], k = in->ndir;
        // every array of the whole batch (len x k per instance), advanced to this shard's first instance
        auto at = [&](const double* const* arr, size_t i, int len) -> const double* {
            return (arr && arr[i]) ? arr[i] + lo * len * k : nullptr;
        };
        std::vector<const double*> p(plen.size()), f(clen.size()), lower(clen.size()), upper(clen.size());
        for (size_t i = 0; i < plen.size(); ++i) p[i] = at(in->p, i, plen[i]);
        for (size_t i = 0; i < clen.size(); ++i) {
            f[i] = at(in->f, i, clen[i]);
            lower[i] = at(in->lower, i, clen[i]);
            upper[i] = at(in->upper, i, clen[i]);
        }
        copra_b200_jvp_in t = *in;
        t.x0 = in->x0 ? in->x0 + lo * nx * k : nullptr;
        t.p = in->p ? p.data() : nullptr;
        t.f = in->f ? f.data() : nullptr;
        t.lower = in->lower ? lower.data() : nullptr;
        t.upper = in->upper ? upper.data() : nullptr;
        return copra_b200_lmpc_jvp(m->h[g], &t, COPRA_B200_HOST, dcontrol ? dcontrol + lo * sz.nU * k : nullptr,
            dtrajectory ? dtrajectory + lo * sz.X * k : nullptr);
    });
}

int copra_b200_multi_lmpc_feedback_gain(copra_b200_multi* m, int steps, double* Ku, double* Kx)
{
    if (!m) return COPRA_B200_E_ARG;
    if (m->lo.size() != m->h.size()) return mfail(m, COPRA_B200_E_STATE, "copra_b200_multi_lmpc_feedback_gain needs a previous run");
    return run_shards(m, [&](int g) {
        copra_b200_sizes sz{};
        int rc = copra_b200_lmpc_built_sizes(m->h[g], &sz);
        if (rc) return rc;
        std::vector<int> plen, clen;
        int nx = 0;
        cb_vjp_lengths(m->h[g], nx, plen, clen);
        const int N = sz.X / nx - 1, nu = N > 0 ? sz.nU / N : 0;
        if (steps < 1 || steps > N) return copra_b200_lmpc_feedback_gain(m->h[g], steps, nullptr, nullptr, COPRA_B200_HOST); // E_ARG
        const long long lo = m->lo[g];
        return copra_b200_lmpc_feedback_gain(m->h[g], steps, Ku ? Ku + lo * nu * steps * nx : nullptr,
            Kx ? Kx + lo * nx * (steps + 1) * nx : nullptr, COPRA_B200_HOST);
    });
}

} // extern "C"
