// BatchedLMPC::initialStateVjp / initialStateJvp (copra_b200_lmpc_vjp_initial_state / _jvp_initial_state) on a small
// initial-state double integrator (C4's shape: target and effort costs, a control bound, an x0 box, R and r): the gradients
// with respect to r, x0lb, x0ub, R and the target against central differences of the controller's own re-solves, the adjoint
// identity between the VJP and the JVP, a symmetric dR, and the errors.  Needs the GPU.
#include <copra/InitialStateLMPC.h>
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

int main()
{
    std::setvbuf(stdout, nullptr, _IONBF, 0);
    const int nx = 2, nu = 1, N = 15, batch = 3, X = nx * (N + 1), nU = nu * N;
    const double T = 0.1;
    Eigen::MatrixXd A(2, 2), B(2, 1), M = Eigen::MatrixXd::Identity(2, 2), Nm = Eigen::MatrixXd::Identity(1, 1);
    Eigen::VectorXd d(2), w(2), wu = Eigen::VectorXd::Constant(1, 1e-2), ud = Eigen::VectorXd::Constant(1, 0.5);
    Eigen::VectorXd ulo(1), uup(1);
    A << 1, T, 0, 1;
    B << 0.5 * T * T, T;
    d << 0.0, -0.02;
    w << 10.0, 100.0;
    ulo << -INFINITY;
    uup << 2.0;
    std::vector<double> x0(nx * batch), xd(nx * batch), R(nx * nx * batch), r(nx * batch), lo(nx * batch), up(nx * batch);
    for (int b = 0; b < batch; ++b) {
        x0[nx * b] = 0.0; x0[nx * b + 1] = -1.0 - 0.3 * b;
        xd[nx * b] = 0.0; xd[nx * b + 1] = -0.5 + 0.2 * b;
        R[nx * nx * b] = 1.0 + 0.2 * b; R[nx * nx * b + 1] = R[nx * nx * b + 2] = 0.1; R[nx * nx * b + 3] = 1.0;
        r[nx * b] = -0.1 * b; r[nx * b + 1] = 0.3;
        lo[nx * b] = -0.1; lo[nx * b + 1] = x0[nx * b + 1] - 0.5;
        up[nx * b] = 0.1; up[nx * b + 1] = x0[nx * b + 1] + 0.5;
    }
    copra::BatchedLMPC ctl(nx, nu, N, batch, true);
    ctl.system(copra::b200::arr(A.data()), copra::b200::arr(B.data()), copra::b200::arr(d.data()), copra::b200::arr(x0.data(), nx));
    ctl.initialStateCost(copra::b200::arr(R.data(), nx * nx), copra::b200::arr(r.data(), nx));
    ctl.initialStateBounds(copra::b200::arr(lo.data(), nx), copra::b200::arr(up.data(), nx));
    copra_b200_cost target{};
    target.kind = COPRA_B200_COST_TARGET; target.rows = 2;
    target.M = copra::b200::arr(M.data()); target.p = copra::b200::arr(xd.data(), nx); target.w = copra::b200::arr(w.data());
    copra_b200_cost effort{};
    effort.kind = COPRA_B200_COST_CONTROL; effort.rows = 1;
    effort.N = copra::b200::arr(Nm.data()); effort.p = copra::b200::arr(ud.data()); effort.w = copra::b200::arr(wu.data());
    copra_b200_constraint cb{};
    cb.kind = COPRA_B200_CSTR_CONTROL_BOUND; cb.rows = nu;
    cb.lower = copra::b200::arr(ulo.data()); cb.upper = copra::b200::arr(uup.data());
    ctl.addCost(target); ctl.addCost(effort);
    ctl.addConstraint(cb);
    REQUIRE(ctl.solve() == batch);

    std::mt19937_64 rng(5);
    std::normal_distribution<double> nrm;
    std::vector<double> dc(size_t(nU) * batch), dt(size_t(X) * batch);
    for (double& v : dc) v = nrm(rng);
    for (double& v : dt) v = nrm(rng);
    auto loss = [&](int b) {
        double v = 0.0;
        for (int i = 0; i < nU; ++i) v += dc[size_t(nU) * b + i] * ctl.controls()[size_t(nU) * b + i];
        for (int i = 0; i < X; ++i) v += dt[size_t(X) * b + i] * ctl.trajectories()[size_t(X) * b + i];
        return v;
    };
    std::vector<double> gx0(nx * batch), gp(nx * batch), gR(nx * nx * batch), gr(nx * batch), glo(nx * batch), gup(nx * batch);
    double* pp[2] = { gp.data(), nullptr };
    copra_b200_vjp_out out{};
    out.x0 = gx0.data(); out.p = pp;
    copra_b200_vjp_initial_out init{ gR.data(), gr.data(), glo.data(), gup.data() };
    ctl.initialStateVjp(dc.data(), dt.data(), out, init);
    for (int b = 0; b < batch; ++b) {
        REQUIRE(gR[nx * nx * b + 1] == gR[nx * nx * b + 2]); // symmetric
        REQUIRE(gx0[nx * b] == 0.0 && gx0[nx * b + 1] == 0.0); // both x0 bounds given: x0 does not enter the build
    }

    // the JVP along random tangents of R, r, x0lb, x0ub and the target, against the VJP (adjoint identity)
    std::vector<double> tR(nx * nx * batch), tr(nx * batch), tlo(nx * batch), tup(nx * batch), tp(nx * batch);
    for (auto* v : { &tR, &tr, &tlo, &tup, &tp })
        for (double& x : *v) x = nrm(rng);
    std::vector<double> ju(size_t(nU) * batch), jx(size_t(X) * batch);
    const double* tpp[2] = { tp.data(), nullptr };
    copra_b200_jvp_in in{};
    in.ndir = 1; in.p = tpp;
    copra_b200_jvp_initial_in tin{ tR.data(), tr.data(), tlo.data(), tup.data() };
    ctl.initialStateJvp(in, tin, ju.data(), jx.data());
    double worst_adj = 0.0;
    for (int b = 0; b < batch; ++b) {
        double lhs = 0.0, rhs = 0.0;
        for (int k = 0; k < nx * nx; ++k) lhs += gR[nx * nx * b + k] * tR[nx * nx * b + k];
        for (int k = 0; k < nx; ++k)
            lhs += gr[nx * b + k] * tr[nx * b + k] + glo[nx * b + k] * tlo[nx * b + k] + gup[nx * b + k] * tup[nx * b + k]
                 + gp[nx * b + k] * tp[nx * b + k];
        for (int i = 0; i < nU; ++i) rhs += dc[size_t(nU) * b + i] * ju[size_t(nU) * b + i];
        for (int i = 0; i < X; ++i) rhs += dt[size_t(X) * b + i] * jx[size_t(X) * b + i];
        worst_adj = std::max(worst_adj, std::fabs(lhs - rhs) / std::max(1.0, std::fabs(rhs)));
    }
    std::printf("[%s] adjoint identity: worst relative difference %.2e\n", worst_adj <= 1e-10 ? " ok " : "FAIL", worst_adj);
    REQUIRE(worst_adj <= 1e-10);

    // central differences of the controller's own re-solves along the same tangent (R moved by its symmetric part)
    std::vector<double> base[5] = { R, r, lo, up, xd };
    std::vector<double>* vars[5] = { &R, &r, &lo, &up, &xd };
    const std::vector<double>* dirs[5] = { &tR, &tr, &tlo, &tup, &tp };
    const double h = 1e-5;
    std::vector<double> lp(batch), lm(batch);
    for (int sg = 0; sg < 2; ++sg) {
        for (int v = 0; v < 5; ++v)
            for (size_t k = 0; k < vars[v]->size(); ++k) {
                double dk = (*dirs[v])[k];
                if (v == 0) { // sym(tR)
                    const size_t b = k / (nx * nx), q = k % (nx * nx), i = q % nx, j = q / nx;
                    dk = 0.5 * ((*dirs[v])[k] + (*dirs[v])[b * nx * nx + j + i * nx]);
                }
                (*vars[v])[k] = base[v][k] + (sg == 0 ? h : -h) * dk;
            }
        REQUIRE(ctl.solve() == batch);
        for (int b = 0; b < batch; ++b) (sg == 0 ? lp : lm)[b] = loss(b);
    }
    double worst = 0.0;
    for (int b = 0; b < batch; ++b) {
        double pred = 0.0;
        for (int i = 0; i < nU; ++i) pred += dc[size_t(nU) * b + i] * ju[size_t(nU) * b + i];
        for (int i = 0; i < X; ++i) pred += dt[size_t(X) * b + i] * jx[size_t(X) * b + i];
        const double est = (lp[b] - lm[b]) / (2.0 * h);
        std::printf("  instance %d: JVP %.12g, central differences %.12g\n", b, pred, est);
        worst = std::max(worst, std::fabs(est - pred) / std::max({ 1.0, std::fabs(est), std::fabs(pred) }));
    }
    std::printf("[%s] worst relative difference to central differences of BatchedLMPC %.2e\n", worst <= 1e-6 ? " ok " : "FAIL", worst);
    REQUIRE(worst <= 1e-6);

    // errors: an LMPC-mode controller throws std::runtime_error
    copra::BatchedLMPC lmpc(nx, nu, N, batch);
    lmpc.system(copra::b200::arr(A.data()), copra::b200::arr(B.data()), copra::b200::arr(d.data()), copra::b200::arr(x0.data(), nx));
    lmpc.addCost(effort);
    REQUIRE(lmpc.solve() == batch);
    bool threw = false;
    try { lmpc.initialStateVjp(dc.data(), nullptr, out, init); } catch (const std::runtime_error&) { threw = true; }
    REQUIRE(threw);
    threw = false;
    try { lmpc.initialStateJvp(in, tin, ju.data(), nullptr); } catch (const std::runtime_error&) { threw = true; }
    REQUIRE(threw);

    std::printf("%d checks, %d failures\n", g_checks, g_fail);
    return g_fail == 0 ? 0 : 1;
}
