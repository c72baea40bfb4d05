// BatchedLMPC::vjp (copra_b200_lmpc_vjp) on a small walk with per-step references and limits, against central differences of
// per-instance copra::LMPC controllers given the same problems as autoSpan'd full-size entries; and its errors.  Needs the GPU.
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

    // the VJP of L = <dc, controls>: gradients batch-major
    std::mt19937_64 rng(7);
    std::normal_distribution<double> nrm;
    std::vector<double> dc(size_t(nU) * batch);
    for (double& v : dc) v = nrm(rng);
    std::vector<double> gx0(nx * batch), gp0(X * batch), gp1(batch), gf(nU * batch), glo1(nU * batch), gup1(nU * batch),
        glo2(X * batch), gup2(X * batch);
    double* pp[2] = { gp0.data(), gp1.data() };
    double* ff[3] = { gf.data(), nullptr, nullptr };
    double* lo[3] = { nullptr, glo1.data(), glo2.data() };
    double* up[3] = { nullptr, gup1.data(), gup2.data() };
    copra_b200_vjp_out out{};
    out.x0 = gx0.data(); out.p = pp; out.f = ff; out.lower = lo; out.upper = up;
    ctl.vjp(dc.data(), nullptr, out);
    double qmax = 0.0; // the lower (Q1) rows must take part for the check below to cover them
    for (double v : glo2) qmax = std::max(qmax, std::fabs(v));
    REQUIRE(qmax > 1e-6);

    // the same controllers one by one (copra::LMPC, autoSpan'd full-size entries): central differences along one random
    // direction per input.  These solves rebuild on the shared engine, so the VJP above is done first.
    struct Input { std::vector<double>* v; size_t off; int len; const std::vector<double>* g; size_t goff; };
    double worst = 0.0;
    int checked = 0;
    for (int b = 0; b < batch; ++b) {
        auto solveOne = [&](Eigen::VectorXd& u) {
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
            if (ok) u = one.control();
            return ok;
        };
        const Input inputs[] = { { &x0, size_t(nx) * b, nx, &gx0, size_t(nx) * b }, { &p, size_t(X) * b, X, &gp0, size_t(X) * b },
            { &ud, 0, 1, &gp1, size_t(b) }, { &f, size_t(nU) * b, nU, &gf, size_t(nU) * b }, { &ulo, 0, nU, &glo1, size_t(nU) * b },
            { &uup, 0, nU, &gup1, size_t(nU) * b }, { &xlo, 0, X, &glo2, size_t(X) * b }, { &xup, 0, X, &gup2, size_t(X) * b } };
        for (const Input& in : inputs) {
            std::vector<double> delta(in.len);
            double pred = 0.0, scale = 1.0;
            for (int k = 0; k < in.len; ++k) {
                const double v = (*in.v)[in.off + k];
                delta[k] = std::isfinite(v) ? nrm(rng) : 0.0;
                pred += (*in.g)[in.goff + k] * delta[k];
                if (std::isfinite(v)) scale = std::max(scale, std::fabs(v));
            }
            const double h = 1e-5 * scale;
            double lval[2] = { 0.0, 0.0 };
            bool ok = true;
            for (int s = 0; s < 2; ++s) {
                const double sg = s == 0 ? 1.0 : -1.0;
                for (int k = 0; k < in.len; ++k) (*in.v)[in.off + k] += sg * h * delta[k];
                Eigen::VectorXd u;
                ok = solveOne(u) && ok;
                for (int k = 0; k < in.len; ++k) (*in.v)[in.off + k] -= sg * h * delta[k];
                if (ok) for (int i = 0; i < nU; ++i) lval[s] += dc[size_t(nU) * b + i] * u(i);
            }
            REQUIRE(ok);
            const double fd = (lval[0] - lval[1]) / (2.0 * h);
            const double err = std::fabs(fd - pred) / std::max({ 1.0, std::fabs(fd), std::fabs(pred) });
            worst = std::max(worst, err);
            ++checked;
        }
    }
    std::printf("[%s] %d directions: worst relative difference of the VJP to central differences of copra::LMPC %.2e\n",
        worst <= 1e-6 ? " ok " : "FAIL", checked, worst);
    REQUIRE(worst <= 1e-6);

    // errors: another controller built on the shared engine since this solve; a full-size cost
    bool threw = false;
    try { ctl.vjp(dc.data(), nullptr, out); } catch (const std::runtime_error&) { threw = true; }
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
    double* pp1[2] = { gp0.data(), gp1.data() };
    double* none[1] = { nullptr };
    copra_b200_vjp_out o2{};
    o2.x0 = gx0.data(); o2.p = pp1; o2.lower = none; o2.upper = none;
    threw = false;
    try { dense.vjp(dc.data(), nullptr, o2); } catch (const std::domain_error&) { threw = true; }
    REQUIRE(threw);
    std::printf("%d checks, %d failures\n", g_checks, g_fail);
    return g_fail == 0 ? 0 : 1;
}
