// BatchedLMPC::vjp with model outputs (copra_b200_lmpc_vjp_model) on a small double integrator with a tracking and an effort
// cost, a control limit (ControlConstraint), control bounds and a trajectory bound whose velocity line has a finite lower
// entry (reference quirk Q1: v <= xlo): dL/dA, dL/dB, dL/dd and the ControlConstraint's dL/dG against central differences of
// per-instance copra::LMPC controllers, the vector gradients bitwise those of the plain vjp, and the errors.  Needs the GPU.
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

static Eigen::MatrixXd spanMat(const Eigen::MatrixXd& m, int n)
{
    Eigen::MatrixXd out = Eigen::MatrixXd::Zero(m.rows() * n, m.cols() * n);
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
    Eigen::MatrixXd A(2, 2), B(2, 1), M = Eigen::MatrixXd::Identity(2, 2), G = Eigen::MatrixXd::Constant(1, 1, 1.0);
    Eigen::MatrixXd Nm = Eigen::MatrixXd::Identity(1, 1);
    Eigen::VectorXd d(2), w(2), wu = Eigen::VectorXd::Constant(1, 1e-2), ud = Eigen::VectorXd::Zero(1), f(1), ulo(1), uup(1);
    Eigen::VectorXd xlo(2), xup(2);
    A << 1, T, 0, 1;
    B << 0.5 * T * T, T;
    d << 0.0, -0.02;
    w << 10.0, 1.0;
    f << 1.6;
    ulo << -2.0;
    uup << 3.0;
    xlo << -INFINITY, 0.4;
    xup << INFINITY, INFINITY;
    std::vector<double> x0(nx * batch), p(nx * batch);
    for (int b = 0; b < batch; ++b) {
        x0[nx * b] = 0.1 * b; x0[nx * b + 1] = -0.2 + 0.05 * b;
        p[nx * b] = 0.5 + 0.3 * b; p[nx * b + 1] = 0.0;
    }
    copra::BatchedLMPC ctl(nx, nu, N, batch);
    ctl.system(copra::b200::arr(A.data()), copra::b200::arr(B.data()), copra::b200::arr(d.data()), copra::b200::arr(x0.data(), nx));
    copra_b200_cost track{};
    track.kind = COPRA_B200_COST_TRAJECTORY; track.rows = 2;
    track.M = copra::b200::arr(M.data()); track.p = copra::b200::arr(p.data(), nx); track.w = copra::b200::arr(w.data());
    copra_b200_cost effort{};
    effort.kind = COPRA_B200_COST_CONTROL; effort.rows = 1;
    effort.N = copra::b200::arr(Nm.data()); effort.p = copra::b200::arr(ud.data()); effort.w = copra::b200::arr(wu.data());
    copra_b200_constraint cc{};
    cc.kind = COPRA_B200_CSTR_CONTROL; cc.rows = 1; cc.is_ineq = 1;
    cc.G = copra::b200::arr(G.data()); cc.f = copra::b200::arr(f.data());
    copra_b200_constraint cb{};
    cb.kind = COPRA_B200_CSTR_CONTROL_BOUND; cb.rows = nu;
    cb.lower = copra::b200::arr(ulo.data()); cb.upper = copra::b200::arr(uup.data());
    copra_b200_constraint tb{};
    tb.kind = COPRA_B200_CSTR_TRAJECTORY_BOUND; tb.rows = nx;
    tb.lower = copra::b200::arr(xlo.data()); tb.upper = copra::b200::arr(xup.data());
    ctl.addCost(track); ctl.addCost(effort);
    ctl.addConstraint(cc); ctl.addConstraint(cb); ctl.addConstraint(tb);
    REQUIRE(ctl.solve() == batch);

    // L = <dc, controls>: the plain vjp, then the same call with the model gradients
    std::mt19937_64 rng(11);
    std::normal_distribution<double> nrm;
    std::vector<double> dc(size_t(nU) * batch);
    for (double& v : dc) v = nrm(rng);
    std::vector<double> gx0(nx * batch), gf(batch), glo(batch * X), gup(batch * X);
    double* none[2] = { nullptr, nullptr };
    double* ff[3] = { gf.data(), nullptr, nullptr };
    double* lo[3] = { nullptr, nullptr, glo.data() };
    double* up[3] = { nullptr, nullptr, gup.data() };
    copra_b200_vjp_out out{};
    out.x0 = gx0.data(); out.p = none; out.f = ff; out.lower = lo; out.upper = up;
    ctl.vjp(dc.data(), nullptr, out);
    const std::vector<double> ref_x0 = gx0, ref_f = gf, ref_lo = glo;
    std::vector<double> dA(nx * nx * batch), dB(nx * nu * batch), dd(nx * batch), dG(batch);
    double* mG[3] = { dG.data(), nullptr, nullptr };
    copra_b200_vjp_model_out mo{};
    mo.A = dA.data(); mo.B = dB.data(); mo.d = dd.data(); mo.G = mG;
    ctl.vjp(dc.data(), nullptr, out, nullptr, mo);
    REQUIRE(gx0 == ref_x0 && gf == ref_f && glo == ref_lo); // one KKT solve, the same vector gradients
    double lmax = 0.0, fmax = 0.0; // the Q1 lower rows and the control limit must be active for the check to cover them
    for (double v : glo) lmax = std::max(lmax, std::fabs(v));
    for (double v : gf) fmax = std::max(fmax, std::fabs(v));
    REQUIRE(lmax > 1e-6 && fmax > 1e-6);

    // errors: an E of a ControlConstraint, a G of a bound (before the per-instance solves below rebuild on the shared engine)
    bool threw = false;
    double* badE[3] = { dG.data(), nullptr, nullptr };
    copra_b200_vjp_model_out bad{};
    bad.E = badE;
    try { ctl.vjp(dc.data(), nullptr, out, nullptr, bad); } catch (const std::domain_error&) { threw = true; }
    REQUIRE(threw);
    threw = false;
    double* badG[3] = { nullptr, dG.data(), nullptr };
    copra_b200_vjp_model_out bad2{};
    bad2.G = badG;
    try { ctl.vjp(dc.data(), nullptr, out, nullptr, bad2); } catch (const std::domain_error&) { threw = true; }
    REQUIRE(threw);

    // per-instance copra::LMPC controllers: central differences along one random direction of A, B, d and G each
    double worst = 0.0;
    int checked = 0;
    for (int b = 0; b < batch; ++b) {
        auto loss = [&](const Eigen::MatrixXd& Ab, const Eigen::MatrixXd& Bb, const Eigen::VectorXd& db, const Eigen::MatrixXd& Gb,
                        double& val) {
            auto ps = std::make_shared<copra::PreviewSystem>(Ab, Bb, db, seg(x0, size_t(nx) * b, nx), N);
            copra::LMPC one(ps);
            auto c1 = std::make_shared<copra::TrajectoryCost>(M, seg(p, size_t(nx) * b, nx));
            auto c2 = std::make_shared<copra::ControlCost>(Nm, ud);
            c1->weights(w); c2->weights(wu);
            auto k1 = std::make_shared<copra::ControlConstraint>(spanMat(Gb, N), Eigen::VectorXd::Constant(nU, f(0)));
            auto k2 = std::make_shared<copra::ControlBoundConstraint>(ulo, uup);
            auto k3 = std::make_shared<copra::TrajectoryBoundConstraint>(xlo, xup);
            one.addCost(c1); one.addCost(c2);
            one.addConstraint(k1); one.addConstraint(k2); one.addConstraint(k3);
            if (!one.solve()) return false;
            const Eigen::VectorXd u = one.control();
            val = 0.0;
            for (int i = 0; i < nU; ++i) val += dc[size_t(nU) * b + i] * u(i);
            return true;
        };
        for (int which = 0; which < 4; ++which) {
            const int len = which == 0 ? nx * nx : which == 1 ? nx * nu : which == 2 ? nx : nu;
            std::vector<double> D(len);
            for (double& v : D) v = nrm(rng);
            const double* g = which == 0 ? dA.data() + nx * nx * b : which == 1 ? dB.data() + nx * nu * b
                            : which == 2 ? dd.data() + nx * b : dG.data() + b;
            double pred = 0.0;
            for (int k = 0; k < len; ++k) pred += g[k] * D[k]; // both column-major
            // central difference, and both one-sided ones: where they disagree the active set moves within the step (a row at
            // its bound with a zero multiplier, or about to reach it) and the solution is not differentiable there
            const double h = 1e-6;
            double v[3] = { 0.0, 0.0, 0.0 };
            bool ok = true;
            for (int sg = 0; sg < 3; ++sg) {
                Eigen::MatrixXd Ap = A, Bp = B, Gp = G;
                Eigen::VectorXd dp = d;
                double* t = which == 0 ? Ap.data() : which == 1 ? Bp.data() : which == 2 ? dp.data() : Gp.data();
                for (int k = 0; k < len; ++k) t[k] += (sg == 0 ? h : sg == 1 ? -h : 0.0) * D[k];
                ok = loss(Ap, Bp, dp, Gp, v[sg]) && ok;
            }
            REQUIRE(ok);
            const double est = (v[0] - v[1]) / (2.0 * h), fwd = (v[0] - v[2]) / h, bwd = (v[2] - v[1]) / h;
            const bool smooth = std::fabs(fwd - bwd) <= 1e-3 * std::max({ 1.0, std::fabs(est) });
            const double err = std::fabs(est - pred) / std::max({ 1.0, std::fabs(est), std::fabs(pred) });
            std::printf("  instance %d, %s: gradient %.12g, central differences %.12g%s\n", b, which == 0 ? "A" : which == 1 ? "B"
                : which == 2 ? "d" : "G", pred, est, smooth ? "" : " (one-sided differences disagree: skipped)");
            if (!smooth) continue;
            worst = std::max(worst, err);
            ++checked;
        }
    }
    REQUIRE(checked >= 12);
    std::printf("[%s] %d directions: worst relative difference of the model gradients to central differences of copra::LMPC %.2e\n",
        worst <= 1e-5 ? " ok " : "FAIL", checked, worst);
    REQUIRE(worst <= 1e-5);

    std::printf("%d checks, %d failures\n", g_checks, g_fail);
    return g_fail == 0 ? 0 : 1;
}
