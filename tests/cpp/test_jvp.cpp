// BatchedLMPC::feedbackGain and BatchedLMPC::jvp (copra_b200_lmpc_feedback_gain / copra_b200_lmpc_jvp) on a small walk with
// per-step references and limits, against central differences of per-instance copra::LMPC controllers given the same problems
// as autoSpan'd full-size entries; and their errors.  Needs the GPU.
#include <copra/LMPC.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <random>
#include <stdexcept>
#include <vector>

static int g_fail = 0, g_checks = 0;
#define REQUIRE(cond)                                                                  \
    do {                                                                               \
        ++g_checks;                                                                    \
        if (!(cond)) { ++g_fail; std::printf("  FAILED %s:%d  %s\n", __FILE__, __LINE__, #cond); } \
    } while (0)

static Eigen::MatrixXd spanMat(const Eigen::MatrixXd& m, int n, int addCols = 0)
{
    Eigen::MatrixXd out = Eigen::MatrixXd::Zero(m.rows() * n, m.cols() * (n + addCols));
    for (int i = 0; i < n; ++i)
        for (int c = 0; c < m.cols(); ++c)
            for (int r = 0; r < m.rows(); ++r) out(i * m.rows() + r, i * m.cols() + c) = m(r, c);
    return out;
}

static Eigen::VectorXd seg(const std::vector<double>& v, size_t off, int n)
{
    Eigen::VectorXd out(n);
    for (int i = 0; i < n; ++i) out(i) = v[off + i];
    return out;
}

int main()
{
    std::setvbuf(stdout, nullptr, _IONBF, 0);
    const int nx = 2, nu = 1, N = 20, batch = 4, X = nx * (N + 1), nU = nu * N;
    const double T = 0.05;
    Eigen::MatrixXd A(2, 2), B(2, 1), M = Eigen::MatrixXd::Identity(2, 2), G = Eigen::MatrixXd::Identity(1, 1);
    Eigen::VectorXd d(2), w(2);
    A << 1, T, 0, 1;
    B << 0.5 * T * T, T;
    d << 0.0, 0.0;
    w << 10.0, 1.0;
    // the vector inputs: x0 and the per-step p of the tracking cost per instance, the control cost's p, the per-step control
    // limit f per instance, per-step control bounds, and a per-step trajectory bound whose velocity line has a finite lower
    // entry (reference quirk Q1: the lower rows are not negated, so it acts as v <= xlo)
    std::vector<double> x0(nx * batch), p(X * batch), ud(1, 0.0), f(nU * batch), ulo(nU), uup(nU), xlo(X), xup(X);
    for (int b = 0; b < batch; ++b) {
        x0[nx * b] = 0.1 * b; x0[nx * b + 1] = -0.2 + 0.05 * b;
        for (int i = 0; i <= N; ++i) { p[size_t(X) * b + nx * i] = std::sin(0.3 * i + b); p[size_t(X) * b + nx * i + 1] = 0.0; }
        for (int i = 0; i < N; ++i) f[size_t(nU) * b + i] = 1.5 + 0.05 * i + 0.1 * b;
    }
    for (int i = 0; i < N; ++i) { ulo[i] = -2.0 - 0.02 * i; uup[i] = 3.0 + 0.01 * i; }
    for (int i = 0; i <= N; ++i) { xlo[nx * i] = xup[nx * i] = INFINITY; xlo[nx * i] = -INFINITY; xlo[nx * i + 1] = 0.4 + 0.01 * i; xup[nx * i + 1] = INFINITY; }

    copra::BatchedLMPC ctl(nx, nu, N, batch);
    ctl.system(copra::b200::arr(A.data()), copra::b200::arr(B.data()), copra::b200::arr(d.data()), copra::b200::arr(x0.data(), nx));
    copra_b200_cost track{};
    track.kind = COPRA_B200_COST_TRAJECTORY; track.rows = 2; track.full_size = COPRA_B200_PER_STEP;
    track.M = copra::b200::arr(M.data()); track.p = copra::b200::arr(p.data(), X); track.w = copra::b200::arr(w.data());
    Eigen::MatrixXd Nm = Eigen::MatrixXd::Identity(1, 1);
    Eigen::VectorXd wu = Eigen::VectorXd::Constant(1, 1e-2);
    copra_b200_cost effort{};
    effort.kind = COPRA_B200_COST_CONTROL; effort.rows = 1;
    effort.N = copra::b200::arr(Nm.data()); effort.p = copra::b200::arr(ud.data()); effort.w = copra::b200::arr(wu.data());
    copra_b200_constraint cc{};
    cc.kind = COPRA_B200_CSTR_CONTROL; cc.rows = 1; cc.is_ineq = 1; cc.full_size = COPRA_B200_PER_STEP;
    cc.G = copra::b200::arr(G.data()); cc.f = copra::b200::arr(f.data(), nU);
    copra_b200_constraint cb{};
    cb.kind = COPRA_B200_CSTR_CONTROL_BOUND; cb.rows = nu; cb.full_size = COPRA_B200_PER_STEP;
    cb.lower = copra::b200::arr(ulo.data()); cb.upper = copra::b200::arr(uup.data());
    copra_b200_constraint tb{};
    tb.kind = COPRA_B200_CSTR_TRAJECTORY_BOUND; tb.rows = nx; tb.full_size = COPRA_B200_PER_STEP;
    tb.lower = copra::b200::arr(xlo.data()); tb.upper = copra::b200::arr(xup.data());
    ctl.addCost(track); ctl.addCost(effort);
    ctl.addConstraint(cc); ctl.addConstraint(cb); ctl.addConstraint(tb);
    REQUIRE(ctl.solve() == batch);

    // the gain over the whole horizon, and one JVP whose direction j moves input j alone (len x k per instance)
    std::vector<double> Ku(size_t(nU) * nx * batch), Kx(size_t(X) * nx * batch);
    ctl.feedbackGain(N, Ku.data(), Kx.data());
    struct Input { std::vector<double>* v; size_t off; int len; bool perInstance; };
    std::mt19937_64 rng(9);
    std::normal_distribution<double> nrm;
    const int k = 8;
    // tangent arrays: x0, p (tracking), p (effort), f, control-bound lower / upper, trajectory-bound lower / upper
    const int lens[k] = { nx, X, 1, nU, nU, nU, X, X };
    std::vector<std::vector<double>> tan(k);
    for (int j = 0; j < k; ++j) tan[j].assign(size_t(lens[j]) * k * batch, 0.0);
    const std::vector<double>* vals[k] = { &x0, &p, &ud, &f, &ulo, &uup, &xlo, &xup };
    const bool per[k] = { true, true, false, true, false, false, false, false };
    for (int b = 0; b < batch; ++b)
        for (int j = 0; j < k; ++j)
            for (int e = 0; e < lens[j]; ++e) {
                const double v = (*vals[j])[(per[j] ? size_t(lens[j]) * b : 0) + e];
                tan[j][(size_t(b) * k + j) * lens[j] + e] = std::isfinite(v) ? nrm(rng) : 0.0;
            }
    const double* tp[2] = { tan[1].data(), tan[2].data() };
    const double* tf[3] = { tan[3].data(), nullptr, nullptr };
    const double* tlo[3] = { nullptr, tan[4].data(), tan[6].data() };
    const double* tup[3] = { nullptr, tan[5].data(), tan[7].data() };
    copra_b200_jvp_in in{};
    in.ndir = k; in.x0 = tan[0].data(); in.p = tp; in.f = tf; in.lower = tlo; in.upper = tup;
    std::vector<double> dU(size_t(nU) * k * batch), dX(size_t(X) * k * batch);
    ctl.jvp(in, dU.data(), dX.data());
    // the first nx rows of Kx are the identity
    double eyeErr = 0.0;
    for (int b = 0; b < batch; ++b)
        for (int s = 0; s < nx; ++s)
            for (int r = 0; r < nx; ++r) eyeErr = std::max(eyeErr, std::fabs(Kx[(size_t(b) * nx + s) * X + r] - (r == s ? 1.0 : 0.0)));
    REQUIRE(eyeErr <= 1e-15);

    // the same controllers one by one (copra::LMPC, autoSpan'd full-size entries).  These solves rebuild on the shared
    // engine, so the batched calls above come first.
    double worstK = 0.0, worstJ = 0.0;
    int checked = 0;
    for (int b = 0; b < batch; ++b) {
        auto solveOne = [&](Eigen::VectorXd& u, Eigen::VectorXd& x) {
            auto ps = std::make_shared<copra::PreviewSystem>(A, B, d, seg(x0, size_t(nx) * b, nx), N);
            copra::LMPC one(ps);
            auto c1 = std::make_shared<copra::TrajectoryCost>(spanMat(M, N + 1), seg(p, size_t(X) * b, X));
            auto c2 = std::make_shared<copra::ControlCost>(Nm, seg(ud, 0, 1));
            c1->weights(w); c2->weights(wu);
            auto k1 = std::make_shared<copra::ControlConstraint>(spanMat(G, N), seg(f, size_t(nU) * b, nU));
            auto k2 = std::make_shared<copra::ControlBoundConstraint>(seg(ulo, 0, nU), seg(uup, 0, nU));
            auto k3 = std::make_shared<copra::TrajectoryBoundConstraint>(seg(xlo, 0, X), seg(xup, 0, X));
            one.addCost(c1); one.addCost(c2);
            one.addConstraint(k1); one.addConstraint(k2); one.addConstraint(k3);
            const bool ok = one.solve();
            if (ok) { u = one.control(); x = one.trajectory(); }
            return ok;
        };
        // central difference of (U, trajectory) along `dir` of input vector `v` (entries off .. off + len)
        auto central = [&](std::vector<double>& v, size_t off, const std::vector<double>& dir, size_t doff, int len, double h,
                           Eigen::VectorXd& gu, Eigen::VectorXd& gx) {
            Eigen::VectorXd u[2], x[2];
            bool ok = true;
            for (int s = 0; s < 2; ++s) {
                const double sg = s == 0 ? 1.0 : -1.0;
                for (int e = 0; e < len; ++e) v[off + e] += sg * h * dir[doff + e];
                ok = solveOne(u[s], x[s]) && ok;
                for (int e = 0; e < len; ++e) v[off + e] -= sg * h * dir[doff + e];
            }
            if (!ok) return false;
            gu = Eigen::VectorXd(u[0].size());
            gx = Eigen::VectorXd(x[0].size());
            for (Eigen::Index r = 0; r < u[0].size(); ++r) gu(r) = (u[0](r) - u[1](r)) / (2.0 * h);
            for (Eigen::Index r = 0; r < x[0].size(); ++r) gx(r) = (x[0](r) - x[1](r)) / (2.0 * h);
            return ok;
        };
        auto relErr = [](const Eigen::VectorXd& fd, const double* got, int len) {
            double e = 0.0, m = 1.0;
            for (int r = 0; r < len; ++r) { e = std::max(e, std::fabs(fd(r) - got[r])); m = std::max({ m, std::fabs(fd(r)), std::fabs(got[r]) }); }
            return e / m;
        };
        // the gain: column s is the tangent along e_s of x0
        for (int s = 0; s < nx; ++s) {
            std::vector<double> es(nx, 0.0);
            es[s] = 1.0;
            Eigen::VectorXd gu, gx;
            const bool ok = central(x0, size_t(nx) * b, es, 0, nx, 1e-5, gu, gx);
            REQUIRE(ok);
            if (!ok) continue;
            worstK = std::max({ worstK, relErr(gu, &Ku[(size_t(b) * nx + s) * nU], nU), relErr(gx, &Kx[(size_t(b) * nx + s) * X], X) });
            ++checked;
        }
        // the JVP, one input per direction
        std::vector<double>* ins[k] = { &x0, &p, &ud, &f, &ulo, &uup, &xlo, &xup };
        for (int j = 0; j < k; ++j) {
            double scale = 1.0;
            const size_t off = per[j] ? size_t(lens[j]) * b : 0;
            for (int e = 0; e < lens[j]; ++e)
                if (std::isfinite((*ins[j])[off + e])) scale = std::max(scale, std::fabs((*ins[j])[off + e]));
            Eigen::VectorXd gu, gx;
            const bool ok = central(*ins[j], off, tan[j], (size_t(b) * k + j) * lens[j], lens[j], 1e-5 * scale, gu, gx);
            REQUIRE(ok);
            if (!ok) continue;
            worstJ = std::max({ worstJ, relErr(gu, &dU[(size_t(b) * k + j) * nU], nU), relErr(gx, &dX[(size_t(b) * k + j) * X], X) });
            ++checked;
        }
    }
    std::printf("[%s] %d directions: worst relative difference to central differences of copra::LMPC: gain %.2e, JVP %.2e\n",
        worstK <= 1e-6 && worstJ <= 1e-6 ? " ok " : "FAIL", checked, worstK, worstJ);
    REQUIRE(worstK <= 1e-6);
    REQUIRE(worstJ <= 1e-6);

    // errors: another controller built on the shared engine since this solve; bad arguments; a full-size cost
    bool threw = false;
    try { ctl.feedbackGain(1, Ku.data(), Kx.data()); } catch (const std::runtime_error&) { threw = true; }
    REQUIRE(threw);
    threw = false;
    try { ctl.jvp(in, dU.data(), dX.data()); } catch (const std::runtime_error&) { threw = true; }
    REQUIRE(threw);
    REQUIRE(ctl.solve() == batch);
    threw = false;
    try { ctl.feedbackGain(0, Ku.data(), Kx.data()); } catch (const std::domain_error&) { threw = true; }
    REQUIRE(threw);
    threw = false;
    try { ctl.feedbackGain(N + 1, Ku.data(), Kx.data()); } catch (const std::domain_error&) { threw = true; }
    REQUIRE(threw);
    copra_b200_jvp_in none = in;
    none.ndir = 0;
    threw = false;
    try { ctl.jvp(none, dU.data(), dX.data()); } catch (const std::domain_error&) { threw = true; }
    REQUIRE(threw);
    copra::BatchedLMPC dense(nx, nu, N, batch);
    dense.system(copra::b200::arr(A.data()), copra::b200::arr(B.data()), copra::b200::arr(d.data()), copra::b200::arr(x0.data(), nx));
    const Eigen::MatrixXd Mfull = spanMat(M, N + 1);
    const Eigen::VectorXd wfull = Eigen::VectorXd::Ones(X);
    copra_b200_cost full{};
    full.kind = COPRA_B200_COST_TRAJECTORY; full.rows = X; full.full_size = 1;
    full.M = copra::b200::arr(Mfull.data()); full.p = copra::b200::arr(p.data(), X); full.w = copra::b200::arr(wfull.data());
    dense.addCost(full); dense.addCost(effort);
    dense.addConstraint(cb);
    REQUIRE(dense.solve() == batch);
    threw = false;
    try { dense.feedbackGain(1, Ku.data(), nullptr); } catch (const std::domain_error&) { threw = true; }
    REQUIRE(threw);
    std::printf("%d checks, %d failures\n", g_checks, g_fail);
    return g_fail == 0 ? 0 : 1;
}
