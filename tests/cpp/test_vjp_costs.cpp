// BatchedLMPC::vjp with cost outputs (copra_b200_lmpc_vjp_costs) on a small double integrator with a tracking, an effort and
// a mixed cost: writes the w / M / N gradients to the file named by argv[1] for tests/test_vjp_costs_gpu.py, which compares
// them with the numpy closed forms of tests/vjp_cost_reference.py; checks here that the vector gradients are bitwise those of
// the plain vjp, and the errors.  Needs the GPU.
#include <copra/LMPC.h>

#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <vector>

static int g_fail = 0, g_checks = 0;
#define REQUIRE(cond)                                                                  \
    do {                                                                               \
        ++g_checks;                                                                    \
        if (!(cond)) { ++g_fail; std::printf("  FAILED %s:%d  %s\n", __FILE__, __LINE__, #cond); } \
    } while (0)

int main(int argc, char** argv)
{
    std::setvbuf(stdout, nullptr, _IONBF, 0);
    if (argc < 2) { std::printf("usage: test_vjp_costs OUTFILE\n"); return 2; }
    const int nx = 2, nu = 1, N = 20, batch = 4, nU = nu * N;
    const double T = 0.05;
    // the problem of tests/test_vjp_costs_gpu.py::_cpp_problem
    Eigen::MatrixXd A(2, 2), B(2, 1), M = Eigen::MatrixXd::Identity(2, 2), Nm = Eigen::MatrixXd::Identity(1, 1);
    Eigen::MatrixXd Mx(1, 2), Nx(1, 1);
    Eigen::VectorXd d = Eigen::VectorXd::Zero(2), w(2), wu(1), wx(1), pu(1), px(1), lo(1), up(1);
    A << 1, T, 0, 1;
    B << 0.5 * T * T, T;
    Mx << 0.5, 1.0;
    Nx << 0.1;
    w << 10.0, 1.0;
    wu << 1e-2;
    wx << 2.0;
    pu << 0.0;
    px << 0.2;
    lo << -2.0;
    up << 3.0;
    std::vector<double> x0(nx * batch), p(nx * batch);
    for (int b = 0; b < batch; ++b) {
        x0[nx * b] = 0.1 * b; x0[nx * b + 1] = -0.2 + 0.05 * b;
        p[nx * b] = std::sin(double(b)); p[nx * b + 1] = 0.0;
    }
    copra::BatchedLMPC ctl(nx, nu, N, batch);
    ctl.system(copra::b200::arr(A.data()), copra::b200::arr(B.data()), copra::b200::arr(d.data()), copra::b200::arr(x0.data(), nx));
    copra_b200_cost track{};
    track.kind = COPRA_B200_COST_TRAJECTORY; track.rows = 2;
    track.M = copra::b200::arr(M.data()); track.p = copra::b200::arr(p.data(), nx); track.w = copra::b200::arr(w.data());
    copra_b200_cost effort{};
    effort.kind = COPRA_B200_COST_CONTROL; effort.rows = 1;
    effort.N = copra::b200::arr(Nm.data()); effort.p = copra::b200::arr(pu.data()); effort.w = copra::b200::arr(wu.data());
    copra_b200_cost mixed{};
    mixed.kind = COPRA_B200_COST_MIXED; mixed.rows = 1;
    mixed.M = copra::b200::arr(Mx.data()); mixed.N = copra::b200::arr(Nx.data()); mixed.p = copra::b200::arr(px.data());
    mixed.w = copra::b200::arr(wx.data());
    copra_b200_constraint cb{};
    cb.kind = COPRA_B200_CSTR_CONTROL_BOUND; cb.rows = nu;
    cb.lower = copra::b200::arr(lo.data()); cb.upper = copra::b200::arr(up.data());
    ctl.addCost(track); ctl.addCost(effort); ctl.addCost(mixed);
    ctl.addConstraint(cb);
    REQUIRE(ctl.solve() == batch);

    // L = <dc, controls>, dc[k] = sin(0.7 k + 1) over the batch-major controls
    std::vector<double> dc(size_t(nU) * batch);
    for (size_t k = 0; k < dc.size(); ++k) dc[k] = std::sin(0.7 * double(k) + 1.0);
    std::vector<double> gx0(nx * batch), gp0(nx * batch), gp1(batch), gp2(batch), glo(batch), gup(batch);
    double* pp[3] = { gp0.data(), gp1.data(), gp2.data() };
    double* none[1] = { nullptr };
    double* lw[1] = { glo.data() };
    double* uw[1] = { gup.data() };
    copra_b200_vjp_out out{};
    out.x0 = gx0.data(); out.p = pp; out.f = none; out.lower = lw; out.upper = uw;
    ctl.vjp(dc.data(), nullptr, out);
    const std::vector<double> ref_x0 = gx0, ref_p0 = gp0, ref_up = gup;

    std::vector<double> dw0(2 * batch), dM0(4 * batch), dw1(batch), dN1(batch), dw2(batch), dM2(2 * batch), dN2(batch);
    double* cw[3] = { dw0.data(), dw1.data(), dw2.data() };
    double* cM[3] = { dM0.data(), nullptr, dM2.data() };
    double* cN[3] = { nullptr, dN1.data(), dN2.data() };
    copra_b200_vjp_cost_out co{};
    co.w = cw; co.M = cM; co.N = cN;
    ctl.vjp(dc.data(), nullptr, out, co);
    REQUIRE(gx0 == ref_x0 && gp0 == ref_p0 && gup == ref_up); // one KKT solve, the same vector gradients
    double mmax = 0.0;
    for (double v : dM2) mmax = std::max(mmax, std::fabs(v));
    REQUIRE(mmax > 0.0);

    FILE* f = std::fopen(argv[1], "w");
    REQUIRE(f != nullptr);
    if (f) {
        for (int b = 0; b < batch; ++b) {
            std::vector<double> row;
            row.insert(row.end(), dw0.begin() + 2 * b, dw0.begin() + 2 * b + 2);
            row.insert(row.end(), dM0.begin() + 4 * b, dM0.begin() + 4 * b + 4);
            row.push_back(dw1[b]); row.push_back(dN1[b]); row.push_back(dw2[b]);
            row.insert(row.end(), dM2.begin() + 2 * b, dM2.begin() + 2 * b + 2);
            row.push_back(dN2[b]);
            for (double v : row) std::fprintf(f, "%.17g ", v);
            std::fprintf(f, "\n");
        }
        std::fclose(f);
    }

    // errors: an N of a TrajectoryCost; another controller built on the shared engine since this solve
    double* badN[3] = { dw0.data(), nullptr, nullptr };
    copra_b200_vjp_cost_out bad{};
    bad.N = badN;
    bool threw = false;
    try { ctl.vjp(dc.data(), nullptr, out, bad); } catch (const std::domain_error&) { threw = true; }
    REQUIRE(threw);
    copra::BatchedLMPC other(nx, nu, N, batch);
    other.system(copra::b200::arr(A.data()), copra::b200::arr(B.data()), copra::b200::arr(d.data()), copra::b200::arr(x0.data(), nx));
    other.addCost(track);
    other.addConstraint(cb);
    REQUIRE(other.solve() == batch);
    threw = false;
    try { ctl.vjp(dc.data(), nullptr, out, co); } catch (const std::runtime_error&) { threw = true; }
    REQUIRE(threw);
    std::printf("%d checks, %d failures\n", g_checks, g_fail);
    return g_fail == 0 ? 0 : 1;
}
