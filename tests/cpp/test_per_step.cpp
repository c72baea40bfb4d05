// BatchedLMPC with per-step references and limits (COPRA_B200_PER_STEP) and its receding-horizon retarget(), against
// per-instance copra::LMPC controllers given the same problems as autoSpan'd full-size entries.  Needs the GPU.
#include <copra/LMPC.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
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
    const int nx = 2, nu = 1, N = 30, batch = 8, X = nx * (N + 1), nU = nu * N;
    const double T = 0.05;
    Eigen::MatrixXd A(2, 2), B(2, 1), M = Eigen::MatrixXd::Identity(2, 2), G = Eigen::MatrixXd::Identity(1, 1);
    Eigen::VectorXd d(2), w(2);
    A << 1, T, 0, 1;
    B << 0.5 * T * T, T;
    d << 0.0, 0.0;
    w << 10.0, 1.0;
    // per instance: a position reference that moves over the horizon, a control limit per step, a velocity bound per step
    std::vector<double> x0(nx * batch), p(X * batch), f(nU * batch), ulo(nU), uup(nU), xlo(X), xup(X);
    auto fill = [&](double shift) {
        for (int b = 0; b < batch; ++b) {
            x0[nx * b] = 0.1 * b - shift; x0[nx * b + 1] = -0.2 + 0.05 * b;
            for (int i = 0; i <= N; ++i) {
                p[size_t(X) * b + nx * i] = std::sin(0.2 * (i + 10 * shift) + b);
                p[size_t(X) * b + nx * i + 1] = 0.0;
            }
            for (int i = 0; i < N; ++i) f[size_t(nU) * b + i] = 2.0 + 0.05 * i + 0.1 * b - shift;
        }
        for (int i = 0; i < N; ++i) { ulo[i] = -3.0 - 0.02 * i + shift; uup[i] = 3.0 + 0.01 * i; }
        for (int i = 0; i <= N; ++i) { xlo[nx * i] = xlo[nx * i + 1] = -INFINITY; xup[nx * i] = INFINITY; xup[nx * i + 1] = 1.5 + 0.01 * i - shift; }
    };
    fill(0.0);
    copra::BatchedLMPC ctl(nx, nu, N, batch);
    ctl.system(copra::b200::arr(A.data()), copra::b200::arr(B.data()), copra::b200::arr(d.data()), copra::b200::arr(x0.data(), nx));
    copra_b200_cost track{};
    track.kind = COPRA_B200_COST_TRAJECTORY; track.rows = 2; track.full_size = COPRA_B200_PER_STEP;
    track.M = copra::b200::arr(M.data()); track.p = copra::b200::arr(p.data(), X); track.w = copra::b200::arr(w.data());
    Eigen::MatrixXd Nm = Eigen::MatrixXd::Identity(1, 1);
    Eigen::VectorXd ud = Eigen::VectorXd::Zero(1), wu = Eigen::VectorXd::Constant(1, 1e-3);
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

    std::vector<std::vector<double>> got;
    REQUIRE(ctl.solve() == batch);
    got.push_back(ctl.controls());
    fill(0.1); // the next tick: new x0, every per-step vector rewritten in place
    REQUIRE(ctl.retarget(copra::b200::arr(x0.data(), nx)) == batch);
    got.push_back(ctl.controls());
    REQUIRE(got[0] != got[1]);

    // references: one copra::LMPC per instance with the autoSpan'd full-size form of the same problem
    for (int k = 0; k < 2; ++k) {
        fill(0.1 * k);
        double worst = 0.0;
        for (int b = 0; b < batch; ++b) {
            auto ps = std::make_shared<copra::PreviewSystem>(A, B, d, seg(x0, size_t(nx) * b, nx), N);
            copra::LMPC one(ps);
            auto c1 = std::make_shared<copra::TrajectoryCost>(spanMat(M, N + 1), seg(p, size_t(X) * b, X));
            auto c2 = std::make_shared<copra::ControlCost>(Nm, ud);
            c1->weights(w); c2->weights(wu);
            auto k1 = std::make_shared<copra::ControlConstraint>(spanMat(G, N), seg(f, size_t(nU) * b, nU));
            auto k2 = std::make_shared<copra::ControlBoundConstraint>(seg(ulo, 0, nU), seg(uup, 0, nU));
            auto k3 = std::make_shared<copra::TrajectoryBoundConstraint>(seg(xlo, 0, X), seg(xup, 0, X));
            one.addCost(c1); one.addCost(c2);
            one.addConstraint(k1); one.addConstraint(k2); one.addConstraint(k3);
            REQUIRE(c1->fullSizeEntry() && k1->fullSizeEntry());
            const bool ok = one.solve();
            REQUIRE(ok);
            if (!ok) continue;
            const Eigen::VectorXd u = one.control();
            double scale = 1.0;
            for (int i = 0; i < nU; ++i) scale = std::max(scale, std::fabs(u(i)));
            for (int i = 0; i < nU; ++i) worst = std::max(worst, std::fabs(got[k][size_t(nU) * b + i] - u(i)) / scale);
        }
        std::printf("[%s] %s: worst control difference to the full-size controllers %.2e\n", worst <= 1e-7 ? " ok " : "FAIL",
            k ? "retarget" : "solve", worst);
        REQUIRE(worst <= 1e-7);
    }
    std::printf("%d checks, %d failures\n", g_checks, g_fail);
    return g_fail == 0 ? 0 : 1;
}
