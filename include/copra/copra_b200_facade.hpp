// copra_b200_facade.hpp -- copra's C++ API surface (namespace copra) on top of the B200 C ABI.
//
// Same class names, argument meaning and error behaviour as the reference so that user code and the
// reference's tests read the same:
//   PreviewSystem                         reference include/PreviewSystem.h:22-68
//   AutoSpan                              include/AutoSpan.h:19-40
//   CostFunction + Trajectory/Target/Control/MixedCost           include/costFunctions.h:22-219
//   Constraint, EqIneqConstraint + Trajectory/Control/Mixed/TrajectoryBound/ControlBound
//                                         include/constraints.h:28-307
//   SolverInterface, SolverFlag, solverFactory                   include/SolverInterface.h:19-81, solverUtils.h:34-67
//   LMPC, InitialStateLMPC                include/LMPC.h:36-191, include/InitialStateLMPC.h:18-42
// New: B200Solver (a SolverInterface backend next to QuadProg/QLD/OSQP/GUROBI) and BatchedLMPC (the
// batched entry point).  All numerics run in the sm_100a kernels behind include/copra_b200.h; this
// header only validates shapes, packs pointers and copies results -- there is no CPU compute path.
//
// Step-size entries use the structured (block-Toeplitz) assembly kernels; full-size (autoSpan'd) entries are
// dense R x X blocks and go through the FP64 tensor-core GEMM (dgemm_dmma.cu).
#pragma once

#if defined(__has_include)
#if __has_include(<Eigen/Core>)
#include <Eigen/Core>
#define COPRA_B200_HAVE_EIGEN 1
#endif
#endif
#ifndef COPRA_B200_HAVE_EIGEN
#include "eigen_shim.hpp"
#endif

#include "../copra_b200.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <limits>
#include <memory>
#include <stdexcept>
#include <atomic>
#include <string>
#include <utility>
#include <vector>

namespace copra {

// ---- error helpers (reference include/debugUtils.h:32-42: exception TYPES are part of the API) ----
#define COPRA_DOMAIN_ERROR(msg) throw std::domain_error(std::string(msg))
#define COPRA_RUNTIME_ERROR(msg) throw std::runtime_error(std::string(msg))

namespace b200 {

// One engine handle PER HOST THREAD (device COPRA_B200_DEVICE, default 0), created on that thread's first use: a handle is not
// thread-safe (include/copra_b200.h), so controllers driven from different threads never share one.
inline copra_b200_handle* handle()
{
    struct Holder {
        copra_b200_handle* h = nullptr;
        Holder()
        {
            copra_b200_options opt{};
            const char* dev = std::getenv("COPRA_B200_DEVICE");
            opt.device = dev ? std::atoi(dev) : 0;
            const int rc = copra_b200_create(&opt, &h);
            if (rc != COPRA_B200_OK)
                COPRA_RUNTIME_ERROR("copra_b200_create failed (" + std::to_string(rc) + "): no usable sm_100 CUDA device; this backend has no CPU fallback");
        }
        ~Holder() { copra_b200_destroy(h); }
    };
    static thread_local Holder holder;
    return holder.h;
}

// Every call that makes this thread's handle hold a different build draws a new epoch (unique across threads);
// controllers remember the epoch of their own build so that lazily fetched getters never read someone else's QP --
// including the QP another thread's handle holds.
inline unsigned long& buildEpoch()
{
    static thread_local unsigned long epoch = 0;
    return epoch;
}
inline unsigned long newEpoch()
{
    static std::atomic<unsigned long> next{ 0 };
    return buildEpoch() = ++next;
}

inline void check(int rc)
{
    if (rc == COPRA_B200_OK) return;
    const std::string msg = copra_b200_last_error(handle());
    if (rc == COPRA_B200_E_ARG) COPRA_DOMAIN_ERROR(msg);
    COPRA_RUNTIME_ERROR("copra_b200 error " + std::to_string(rc) + ": " + msg);
}

inline copra_b200_array arr(const double* p, long long stride = 0)
{
    copra_b200_array a;
    a.ptr = p;
    a.stride = stride;
    return a;
}

} // namespace b200

// ====================================================================================================
// AutoSpan (host-side helper, reference src/AutoSpan.cpp:10-47)
// ====================================================================================================
struct AutoSpan {
    AutoSpan() = delete;
    static void spanMatrix(Eigen::MatrixXd& mat, Eigen::Index new_dim, int addCols = 0)
    {
        const Eigen::Index rows = mat.rows();
        if (new_dim == rows) return;
        const Eigen::Index cols = mat.cols();
        const Eigen::Index steps = rows > 0 ? new_dim / rows : 0;
        if (steps * rows != new_dim) COPRA_DOMAIN_ERROR("spanMatrix: new dimension is not a multiple of the matrix rows");
        Eigen::MatrixXd out = Eigen::MatrixXd::Zero(new_dim, cols * (steps + addCols));
        for (Eigen::Index s = 0; s < steps; ++s)
            for (Eigen::Index c = 0; c < cols; ++c)
                for (Eigen::Index r = 0; r < rows; ++r) out(s * rows + r, s * cols + c) = mat(r, c);
        mat = out;
    }
    static void spanVector(Eigen::VectorXd& vec, Eigen::Index new_dim)
    {
        const Eigen::Index rows = vec.rows();
        if (new_dim == rows) return;
        const Eigen::Index steps = rows > 0 ? new_dim / rows : 0;
        if (steps * rows != new_dim) COPRA_DOMAIN_ERROR("spanVector: new dimension is not a multiple of the vector rows");
        Eigen::VectorXd out(new_dim);
        for (Eigen::Index s = 0; s < steps; ++s)
            for (Eigen::Index r = 0; r < rows; ++r) out(s * rows + r) = vec(r);
        vec = out;
    }
};

// ====================================================================================================
// PreviewSystem
// ====================================================================================================
struct PreviewSystem {
    PreviewSystem() = default;
    PreviewSystem(const Eigen::MatrixXd& state, const Eigen::MatrixXd& control, const Eigen::VectorXd& bias,
        const Eigen::VectorXd& xInit, int numberOfSteps)
    {
        system(state, control, bias, xInit, numberOfSteps);
    }

    // dimension checks of src/PreviewSystem.cpp:19-33 (std::domain_error), allocation :35-54
    void system(const Eigen::MatrixXd& state, const Eigen::MatrixXd& control, const Eigen::VectorXd& bias,
        const Eigen::VectorXd& xInit, int numberOfSteps)
    {
        if (xInit.rows() != state.rows()) COPRA_DOMAIN_ERROR("xInit and state should have the same number of rows");
        if (state.rows() != state.cols()) COPRA_DOMAIN_ERROR("state should be a square matrix");
        if (xInit.rows() != control.rows()) COPRA_DOMAIN_ERROR("xInit and control should have the same number of rows");
        if (xInit.rows() != bias.rows()) COPRA_DOMAIN_ERROR("xInit and bias should have the same number of rows");
        if (numberOfSteps <= 0) COPRA_DOMAIN_ERROR("The number of step sould be a positive number! ");
        isUpdated = false;
        nrUStep = numberOfSteps;
        nrXStep = numberOfSteps + 1;
        xDim = static_cast<int>(state.cols());
        uDim = static_cast<int>(control.cols());
        fullXDim = xDim * nrXStep;
        fullUDim = uDim * nrUStep;
        x0 = xInit; A = state; B = control; d = bias;
        Phi = Eigen::MatrixXd::Zero(fullXDim, xDim);
        for (int i = 0; i < xDim; ++i) Phi(i, i) = 1.0;
        Psi = Eigen::MatrixXd::Zero(fullXDim, fullUDim);
        xi = Eigen::VectorXd::Zero(fullXDim);
    }

    // K1 on the GPU (replaces src/PreviewSystem.cpp:57-74)
    void updateSystem()
    {
        b200::check(copra_b200_condense(b200::handle(), xDim, uDim, nrUStep, 1, b200::arr(A.data()), b200::arr(B.data()),
            b200::arr(d.data()), Phi.data(), Psi.data(), xi.data(), COPRA_B200_HOST));
        b200::newEpoch();
        isUpdated = true;
    }

    void xInit(const Eigen::VectorXd& xInit)
    {
        if (xInit.rows() != x0.rows()) COPRA_DOMAIN_ERROR("xInit has a bad dimension");
        x0 = xInit;
    }

    bool isUpdated = false;
    int nrUStep = 0, nrXStep = 0, xDim = 0, uDim = 0, fullXDim = 0, fullUDim = 0;
    Eigen::VectorXd x0;
    Eigen::MatrixXd A, B;
    Eigen::VectorXd d;
    Eigen::MatrixXd Phi, Psi;
    Eigen::VectorXd xi;
};

namespace b200 {

// A batch-of-one problem description under construction (keeps the descriptor arrays alive).
struct Description {
    copra_b200_problem p{};
    std::vector<copra_b200_cost> costs;
    std::vector<copra_b200_constraint> cstrs;
    void system(const PreviewSystem& ps)
    {
        p.nx = ps.xDim; p.nu = ps.uDim; p.N = ps.nrUStep; p.batch = 1;
        p.A = arr(ps.A.data()); p.B = arr(ps.B.data()); p.d = arr(ps.d.data()); p.x0 = arr(ps.x0.data());
        p.memory = COPRA_B200_HOST;
    }
    const copra_b200_problem* finish()
    {
        p.ncost = int(costs.size()); p.costs = costs.data();
        p.ncstr = int(cstrs.size()); p.cstrs = cstrs.data();
        return &p;
    }
};

inline void download(int what, Eigen::MatrixXd& out, Eigen::Index r, Eigen::Index c)
{
    out.resize(r, c);
    if (r * c > 0) check(copra_b200_lmpc_download(handle(), what, out.data(), COPRA_B200_HOST));
}
inline void download(int what, Eigen::VectorXd& out, Eigen::Index n)
{
    out.resize(n);
    if (n > 0) check(copra_b200_lmpc_download(handle(), what, out.data(), COPRA_B200_HOST));
}

} // namespace b200

// ====================================================================================================
// Cost functions
// ====================================================================================================
class CostFunction {
public:
    explicit CostFunction(std::string&& name) : name_(std::move(name)), fullSizeEntry_(false) {}
    virtual ~CostFunction() = default;
    virtual void autoSpan() {}
    virtual void initializeCost(const PreviewSystem& ps)
    {
        Q_.resize(ps.fullUDim, ps.fullUDim);
        c_.resize(ps.fullUDim);
        E_.resize(ps.xDim, ps.fullUDim);
        f_.resize(ps.fullUDim);
    }
    // Evaluate this cost alone on the GPU (K1 + K2 with one cost family): Q(), c(), E(), f().
    virtual void update(const PreviewSystem& ps)
    {
        b200::Description D;
        D.system(ps);
        D.p.flags = COPRA_B200_FLAG_NO_REG;
        D.costs.push_back(describe());
        b200::check(copra_b200_lmpc_build(b200::handle(), D.finish()));
        b200::newEpoch();
        b200::download(COPRA_B200_GET_Q, Q_, ps.fullUDim, ps.fullUDim);
        b200::download(COPRA_B200_GET_C, c_, ps.fullUDim);
        b200::download(COPRA_B200_GET_COST_E, E_, ps.xDim, ps.fullUDim);
        b200::download(COPRA_B200_GET_COST_F, f_, ps.fullUDim);
    }
    // weights(): assign or tile (include/costFunctions.h:54-67)
    void weights(const Eigen::VectorXd& w)
    {
        if (w.rows() == weights_.rows()) weights_ = w;
        else if (w.rows() > 0 && weights_.rows() % w.rows() == 0) {
            for (Eigen::Index i = 0; i < weights_.rows() / w.rows(); ++i)
                for (Eigen::Index k = 0; k < w.rows(); ++k) weights_(i * w.rows() + k) = w(k);
        } else COPRA_DOMAIN_ERROR("weights should have " + std::to_string(weights_.rows()) + " rows (or a divisor of it)");
    }
    template <typename T, typename = typename std::enable_if<std::is_arithmetic<T>::value>::type> void weight(T w)
    {
        weights_.setConstant(double(w));
    }
    const std::string& name() const noexcept { return name_; }
    const Eigen::MatrixXd& Q() const noexcept { return Q_; }
    const Eigen::VectorXd& c() const noexcept { return c_; }
    const Eigen::MatrixXd& E() const noexcept { return E_; }
    const Eigen::VectorXd& f() const noexcept { return f_; }
    bool fullSizeEntry() const noexcept { return fullSizeEntry_; }
    virtual copra_b200_cost describe() const = 0; // C-ABI descriptor (step-size entries)

protected:
    std::string name_;
    bool fullSizeEntry_;
    Eigen::MatrixXd Q_, E_;
    Eigen::VectorXd c_, f_, weights_;
};

class TrajectoryCost final : public CostFunction {
public:
    TrajectoryCost(Eigen::MatrixXd M, Eigen::VectorXd p) : CostFunction("TrajectoryCost"), M_(std::move(M)), p_(std::move(p))
    {
        weights_ = Eigen::VectorXd::Ones(p_.rows());
    }
    void autoSpan() override // src/costFunctions.cpp:36-42
    {
        const Eigen::Index md = std::max(M_.rows(), std::max(weights_.rows(), p_.rows()));
        AutoSpan::spanMatrix(M_, md);
        AutoSpan::spanVector(p_, md);
        AutoSpan::spanVector(weights_, md);
    }
    void initializeCost(const PreviewSystem& ps) override // :44-61
    {
        CostFunction::initializeCost(ps);
        if (M_.rows() != p_.rows()) COPRA_DOMAIN_ERROR("M and p should have the same number of rows (try autoSpan)");
        if (M_.cols() == ps.xDim) fullSizeEntry_ = false;
        else if (M_.cols() == ps.fullXDim) fullSizeEntry_ = true;
        else COPRA_DOMAIN_ERROR("M should have xDim or fullXDim columns");
    }
    copra_b200_cost describe() const override
    {
        copra_b200_cost c{};
        c.kind = COPRA_B200_COST_TRAJECTORY; c.rows = int(M_.rows()); c.full_size = fullSizeEntry_;
        c.M = b200::arr(M_.data()); c.p = b200::arr(p_.data()); c.w = b200::arr(weights_.data());
        return c;
    }

private:
    Eigen::MatrixXd M_;
    Eigen::VectorXd p_;
};

class TargetCost final : public CostFunction {
public:
    TargetCost(Eigen::MatrixXd M, Eigen::VectorXd p) : CostFunction("TargetCost"), M_(std::move(M)), p_(std::move(p))
    {
        weights_ = Eigen::VectorXd::Ones(p_.rows());
    }
    void initializeCost(const PreviewSystem& ps) override // :88-98
    {
        CostFunction::initializeCost(ps);
        if (M_.rows() != p_.rows()) COPRA_DOMAIN_ERROR("M and p should have the same number of rows");
        if (M_.cols() != ps.xDim) COPRA_DOMAIN_ERROR("M should have xDim columns");
    }
    copra_b200_cost describe() const override
    {
        copra_b200_cost c{};
        c.kind = COPRA_B200_COST_TARGET; c.rows = int(M_.rows());
        c.M = b200::arr(M_.data()); c.p = b200::arr(p_.data()); c.w = b200::arr(weights_.data());
        return c;
    }

private:
    Eigen::MatrixXd M_;
    Eigen::VectorXd p_;
};

class ControlCost final : public CostFunction {
public:
    ControlCost(Eigen::MatrixXd N, Eigen::VectorXd p) : CostFunction("ControlCost"), N_(std::move(N)), p_(std::move(p))
    {
        weights_ = Eigen::VectorXd::Ones(p_.rows());
    }
    void autoSpan() override // :114-120
    {
        const Eigen::Index md = std::max(N_.rows(), std::max(weights_.rows(), p_.rows()));
        AutoSpan::spanMatrix(N_, md);
        AutoSpan::spanVector(p_, md);
        AutoSpan::spanVector(weights_, md);
    }
    void initializeCost(const PreviewSystem& ps) override // :122-137
    {
        CostFunction::initializeCost(ps);
        if (N_.rows() != p_.rows()) COPRA_DOMAIN_ERROR("N and p should have the same number of rows (try autoSpan)");
        if (N_.cols() == ps.uDim) fullSizeEntry_ = false;
        else if (N_.cols() == ps.fullUDim) fullSizeEntry_ = true;
        else COPRA_DOMAIN_ERROR("N should have uDim or fullUDim columns");
    }
    copra_b200_cost describe() const override
    {
        copra_b200_cost c{};
        c.kind = COPRA_B200_COST_CONTROL; c.rows = int(N_.rows()); c.full_size = fullSizeEntry_;
        c.N = b200::arr(N_.data()); c.p = b200::arr(p_.data()); c.w = b200::arr(weights_.data());
        return c;
    }

private:
    Eigen::MatrixXd N_;
    Eigen::VectorXd p_;
};

class MixedCost final : public CostFunction {
public:
    MixedCost(Eigen::MatrixXd M, Eigen::MatrixXd N, Eigen::VectorXd p)
        : CostFunction("MixedCost"), M_(std::move(M)), N_(std::move(N)), p_(std::move(p))
    {
        weights_ = Eigen::VectorXd::Ones(p_.rows());
    }
    void autoSpan() override // :164-171 (M gets one extra zero block column)
    {
        const Eigen::Index md = std::max(M_.rows(), std::max(N_.rows(), std::max(weights_.rows(), p_.rows())));
        AutoSpan::spanMatrix(M_, md, 1);
        AutoSpan::spanMatrix(N_, md);
        AutoSpan::spanVector(p_, md);
        AutoSpan::spanVector(weights_, md);
    }
    void initializeCost(const PreviewSystem& ps) override // :173-193
    {
        CostFunction::initializeCost(ps);
        if (M_.rows() != p_.rows()) COPRA_DOMAIN_ERROR("M and p should have the same number of rows (try autoSpan)");
        if (N_.rows() != p_.rows()) COPRA_DOMAIN_ERROR("N and p should have the same number of rows (try autoSpan)");
        if (M_.cols() == ps.xDim && N_.cols() == ps.uDim) fullSizeEntry_ = false;
        else if (M_.cols() == ps.fullXDim && N_.cols() == ps.fullUDim) fullSizeEntry_ = true;
        else COPRA_DOMAIN_ERROR("M / N should have (xDim, uDim) or (fullXDim, fullUDim) columns");
    }
    copra_b200_cost describe() const override
    {
        copra_b200_cost c{};
        c.kind = COPRA_B200_COST_MIXED; c.rows = int(M_.rows()); c.full_size = fullSizeEntry_;
        c.M = b200::arr(M_.data()); c.N = b200::arr(N_.data()); c.p = b200::arr(p_.data()); c.w = b200::arr(weights_.data());
        return c;
    }

private:
    Eigen::MatrixXd M_, N_;
    Eigen::VectorXd p_;
};

// ====================================================================================================
// Constraints
// ====================================================================================================
enum class ConstraintFlag { Constraint, EqualityConstraint, InequalityConstraint, BoundConstraint };

class Constraint {
public:
    explicit Constraint(std::string&& name) : name_(std::move(name)), nrConstr_(0), fullSizeEntry_(false), hasBeenInitialized_(false) {}
    virtual ~Constraint() = default;
    virtual void autoSpan() = 0;
    virtual void initializeConstraint(const PreviewSystem& ps) = 0;
    virtual void update(const PreviewSystem& ps) = 0;
    virtual ConstraintFlag constraintType() const noexcept = 0;
    const std::string& name() const noexcept { return name_; }
    int nrConstr() noexcept { return nrConstr_; }
    bool fullSizeEntry() const noexcept { return fullSizeEntry_; }
    virtual copra_b200_constraint describe() const = 0;

protected:
    std::string name_;
    int nrConstr_;
    bool fullSizeEntry_;
    bool hasBeenInitialized_;
};

class EqIneqConstraint : public Constraint {
public:
    EqIneqConstraint(const std::string& qualifier, bool isInequalityConstraint)
        : Constraint(qualifier + (isInequalityConstraint ? " inequality constraint" : " equality constraint")), isIneq_(isInequalityConstraint)
    {
    }
    const Eigen::MatrixXd& A() { return A_; }
    const Eigen::VectorXd& b() { return b_; }
    const Eigen::MatrixXd& Y() { return Y_; }
    const Eigen::VectorXd& z() { return z_; }
    // Evaluate this constraint alone on the GPU (K1 + K3 + K4 with one family): A(), b(), Y(), z().
    void update(const PreviewSystem& ps) override
    {
        b200::Description D;
        D.system(ps);
        D.cstrs.push_back(describe());
        b200::check(copra_b200_lmpc_build(b200::handle(), D.finish()));
        b200::newEpoch();
        const bool eq = constraintType() == ConstraintFlag::EqualityConstraint;
        b200::download(eq ? COPRA_B200_GET_AEQ : COPRA_B200_GET_AINEQ, A_, nrConstr_, ps.fullUDim);
        b200::download(eq ? COPRA_B200_GET_BEQ : COPRA_B200_GET_BINEQ, b_, nrConstr_);
        b200::download(eq ? COPRA_B200_GET_YEQ : COPRA_B200_GET_YINEQ, Y_, nrConstr_, ps.xDim);
        b200::download(eq ? COPRA_B200_GET_ZEQ : COPRA_B200_GET_ZINEQ, z_, nrConstr_);
    }

protected:
    void allocate(const PreviewSystem& ps)
    {
        A_.resize(nrConstr_, ps.fullUDim);
        b_.resize(nrConstr_);
        Y_.resize(nrConstr_, ps.xDim);
        z_.resize(nrConstr_);
    }
    Eigen::MatrixXd A_, Y_;
    Eigen::VectorXd b_, z_;
    bool isIneq_;
};

class TrajectoryConstraint final : public EqIneqConstraint {
public:
    TrajectoryConstraint(Eigen::MatrixXd E, Eigen::VectorXd f, bool isInequalityConstraint = true)
        : EqIneqConstraint("Trajectory", isInequalityConstraint), E_(std::move(E)), f_(std::move(f))
    {
    }
    void autoSpan() override // src/constraints.cpp:38-43
    {
        const Eigen::Index md = std::max(E_.rows(), f_.rows());
        AutoSpan::spanMatrix(E_, md);
        AutoSpan::spanVector(f_, md);
    }
    void initializeConstraint(const PreviewSystem& ps) override // :45-64
    {
        if (E_.rows() != f_.rows()) COPRA_DOMAIN_ERROR("E and f should have the same number of rows (try autoSpan)");
        if (E_.cols() == ps.xDim) { fullSizeEntry_ = false; nrConstr_ = int(E_.rows()) * ps.nrXStep; }
        else if (E_.cols() == ps.fullXDim) { fullSizeEntry_ = true; nrConstr_ = int(E_.rows()); }
        else COPRA_DOMAIN_ERROR("E should have xDim or fullXDim columns");
        allocate(ps);
    }
    ConstraintFlag constraintType() const noexcept override
    {
        return isIneq_ ? ConstraintFlag::InequalityConstraint : ConstraintFlag::EqualityConstraint;
    }
    copra_b200_constraint describe() const override
    {
        copra_b200_constraint c{};
        c.kind = COPRA_B200_CSTR_TRAJECTORY; c.rows = int(E_.rows()); c.is_ineq = isIneq_; c.full_size = fullSizeEntry_;
        c.E = b200::arr(E_.data()); c.f = b200::arr(f_.data());
        return c;
    }

private:
    Eigen::MatrixXd E_;
    Eigen::VectorXd f_;
};

class ControlConstraint final : public EqIneqConstraint {
public:
    ControlConstraint(Eigen::MatrixXd G, Eigen::VectorXd f, bool isInequalityConstraint = true)
        : EqIneqConstraint("Control", isInequalityConstraint), G_(std::move(G)), f_(std::move(f))
    {
    }
    void autoSpan() override // :99-104
    {
        const Eigen::Index md = std::max(G_.rows(), f_.rows());
        AutoSpan::spanMatrix(G_, md);
        AutoSpan::spanVector(f_, md);
    }
    void initializeConstraint(const PreviewSystem& ps) override // :106-135 (quirk Q9: single initialisation)
    {
        if (hasBeenInitialized_) COPRA_RUNTIME_ERROR("You have initialized a ControlConstraint twice. As move semantics are used, you can't do so.");
        if (G_.rows() != f_.rows()) COPRA_DOMAIN_ERROR("G and f should have the same number of rows (try autoSpan)");
        if (G_.cols() == ps.uDim) { fullSizeEntry_ = false; nrConstr_ = int(G_.rows()) * ps.nrUStep; }
        else if (G_.cols() == ps.fullUDim) { fullSizeEntry_ = true; nrConstr_ = int(G_.rows()); }
        else COPRA_DOMAIN_ERROR("G should have uDim or fullUDim columns");
        allocate(ps);
        hasBeenInitialized_ = true;
    }
    ConstraintFlag constraintType() const noexcept override
    {
        return isIneq_ ? ConstraintFlag::InequalityConstraint : ConstraintFlag::EqualityConstraint;
    }
    copra_b200_constraint describe() const override
    {
        copra_b200_constraint c{};
        c.kind = COPRA_B200_CSTR_CONTROL; c.rows = int(G_.rows()); c.is_ineq = isIneq_; c.full_size = fullSizeEntry_;
        c.G = b200::arr(G_.data()); c.f = b200::arr(f_.data());
        return c;
    }

private:
    Eigen::MatrixXd G_;
    Eigen::VectorXd f_;
};

class MixedConstraint final : public EqIneqConstraint {
public:
    MixedConstraint(Eigen::MatrixXd E, Eigen::MatrixXd G, Eigen::VectorXd f, bool isInequalityConstraint = true)
        : EqIneqConstraint("Control", isInequalityConstraint) // sic: the reference names it "Control" (quirk Q10)
        , E_(std::move(E)), G_(std::move(G)), f_(std::move(f))
    {
    }
    void autoSpan() override // :163-169
    {
        const Eigen::Index md = std::max(f_.rows(), std::max(E_.rows(), G_.rows()));
        AutoSpan::spanMatrix(E_, md, 1);
        AutoSpan::spanMatrix(G_, md);
        AutoSpan::spanVector(f_, md);
    }
    void initializeConstraint(const PreviewSystem& ps) override // :171-195
    {
        if (E_.rows() != f_.rows()) COPRA_DOMAIN_ERROR("E and f should have the same number of rows (try autoSpan)");
        if (G_.rows() != f_.rows()) COPRA_DOMAIN_ERROR("G and f should have the same number of rows (try autoSpan)");
        if (E_.cols() == ps.xDim && G_.cols() == ps.uDim) { fullSizeEntry_ = false; nrConstr_ = int(E_.rows()) * ps.nrUStep; }
        else if (E_.cols() == ps.fullXDim && G_.cols() == ps.fullUDim) { fullSizeEntry_ = true; nrConstr_ = int(E_.rows()); }
        else COPRA_DOMAIN_ERROR("E / G should have (xDim, uDim) or (fullXDim, fullUDim) columns");
        allocate(ps);
    }
    ConstraintFlag constraintType() const noexcept override
    {
        return isIneq_ ? ConstraintFlag::InequalityConstraint : ConstraintFlag::EqualityConstraint;
    }
    copra_b200_constraint describe() const override
    {
        copra_b200_constraint c{};
        c.kind = COPRA_B200_CSTR_MIXED; c.rows = int(E_.rows()); c.is_ineq = isIneq_; c.full_size = fullSizeEntry_;
        c.E = b200::arr(E_.data()); c.G = b200::arr(G_.data()); c.f = b200::arr(f_.data());
        return c;
    }

private:
    Eigen::MatrixXd E_, G_;
    Eigen::VectorXd f_;
};

class TrajectoryBoundConstraint final : public EqIneqConstraint {
public:
    TrajectoryBoundConstraint(Eigen::VectorXd lower, Eigen::VectorXd upper)
        : EqIneqConstraint("Trajectory bound", true), lower_(std::move(lower)), upper_(std::move(upper))
    {
        selectLines(true, true); // include/constraints.h:247-254
    }
    void autoSpan() override // :241-261 (the re-selection there is dead code: both vectors have max_dim rows by then)
    {
        const Eigen::Index md = std::max(lower_.rows(), upper_.rows());
        AutoSpan::spanVector(lower_, md);
        AutoSpan::spanVector(upper_, md);
        if (lower_.rows() != md) selectLines(true, false);
        if (upper_.rows() != md) selectLines(false, true);
    }
    void initializeConstraint(const PreviewSystem& ps) override // :263-282
    {
        if (lower_.rows() != upper_.rows()) COPRA_DOMAIN_ERROR("lower and upper should have the same number of rows (try autoSpan)");
        const int lines = int(lowerLines_.size() + upperLines_.size());
        if (lower_.rows() == ps.xDim) { fullSizeEntry_ = false; nrConstr_ = lines * ps.nrXStep; }
        else if (lower_.rows() == ps.fullXDim) { fullSizeEntry_ = true; nrConstr_ = lines; }
        else COPRA_DOMAIN_ERROR("lower / upper should have xDim or fullXDim rows");
        allocate(ps);
        // The C ABI selects the finite lines itself.  After autoSpan() the reference keeps the line lists of the
        // UN-spanned vectors (the re-selection at src/constraints.cpp:246-260 is dead code), so the vectors handed to
        // the engine are masked to exactly lowerLines_ / upperLines_.
        const double inf = std::numeric_limits<double>::infinity();
        lowerSel_ = Eigen::VectorXd::Constant(lower_.rows(), -inf);
        upperSel_ = Eigen::VectorXd::Constant(upper_.rows(), inf);
        for (int l : lowerLines_) lowerSel_(l) = lower_(l);
        for (int l : upperLines_) upperSel_(l) = upper_(l);
    }
    ConstraintFlag constraintType() const noexcept override { return ConstraintFlag::InequalityConstraint; }
    copra_b200_constraint describe() const override
    {
        copra_b200_constraint c{};
        c.kind = COPRA_B200_CSTR_TRAJECTORY_BOUND; c.rows = int(lower_.rows()); c.is_ineq = 1; c.full_size = fullSizeEntry_;
        c.lower = b200::arr(lowerSel_.data()); c.upper = b200::arr(upperSel_.data());
        return c;
    }

private:
    void selectLines(bool lo, bool up)
    {
        const double inf = std::numeric_limits<double>::infinity();
        if (lo) {
            lowerLines_.clear();
            for (int l = 0; l < lower_.rows(); ++l) if (lower_(l) != -inf) lowerLines_.push_back(l);
        }
        if (up) {
            upperLines_.clear();
            for (int l = 0; l < upper_.rows(); ++l) if (upper_(l) != inf) upperLines_.push_back(l);
        }
    }
    Eigen::VectorXd lower_, upper_, lowerSel_, upperSel_;
    std::vector<int> lowerLines_, upperLines_;
};

class ControlBoundConstraint final : public Constraint {
public:
    ControlBoundConstraint(Eigen::VectorXd lower, Eigen::VectorXd upper)
        : Constraint("Control bound constraint"), lower_(std::move(lower)), upper_(std::move(upper))
    {
    }
    void autoSpan() override // :326-331
    {
        const Eigen::Index md = std::max(lower_.rows(), upper_.rows());
        AutoSpan::spanVector(lower_, md);
        AutoSpan::spanVector(upper_, md);
    }
    void initializeConstraint(const PreviewSystem& ps) override // :333-357 (quirk Q9)
    {
        if (hasBeenInitialized_) COPRA_RUNTIME_ERROR("You have initialized a ControlBoundConstraint twice. As move semantics are used, you can't do so.");
        if (lower_.rows() != upper_.rows()) COPRA_DOMAIN_ERROR("lower and upper should have the same number of rows (try autoSpan)");
        if (lower_.rows() == ps.uDim) { fullSizeEntry_ = false; nrConstr_ = ps.fullUDim; }
        else if (lower_.rows() == ps.fullUDim) { fullSizeEntry_ = true; nrConstr_ = int(lower_.rows()); }
        else COPRA_DOMAIN_ERROR("lower / upper should have uDim or fullUDim rows");
        lb_.resize(nrConstr_);
        ub_.resize(nrConstr_);
        hasBeenInitialized_ = true;
    }
    void update(const PreviewSystem& ps) override // :359-367 -- a pure tiling, no arithmetic
    {
        const Eigen::Index reps = fullSizeEntry_ ? 1 : ps.nrUStep, len = lower_.rows();
        for (Eigen::Index i = 0; i < reps; ++i)
            for (Eigen::Index k = 0; k < len; ++k) { lb_(i * len + k) = lower_(k); ub_(i * len + k) = upper_(k); }
    }
    ConstraintFlag constraintType() const noexcept override { return ConstraintFlag::BoundConstraint; }
    const Eigen::VectorXd& lower() { return lb_; }
    const Eigen::VectorXd& upper() { return ub_; }
    copra_b200_constraint describe() const override
    {
        copra_b200_constraint c{};
        c.kind = COPRA_B200_CSTR_CONTROL_BOUND; c.rows = int(lower_.rows()); c.full_size = fullSizeEntry_;
        c.lower = b200::arr(lower_.data()); c.upper = b200::arr(upper_.data());
        return c;
    }

private:
    Eigen::VectorXd lower_, upper_, lb_, ub_;
};

// ====================================================================================================
// Solver plug-in boundary
// ====================================================================================================
class SolverInterface {
public:
    SolverInterface() = default;
    virtual ~SolverInterface() = default;
    virtual int SI_fail() const = 0;
    virtual void SI_inform() const = 0;
    virtual int SI_iter() const { std::cout << "No iter() function for this qp" << std::endl; return 0; }
    virtual int SI_maxIter() const { std::cout << "No maxIter() function for this qp" << std::endl; return 0; }
    virtual void SI_maxIter(int) { std::cout << "No maxIter(int) function for this qp" << std::endl; }
    virtual void SI_printLevel(int) { std::cout << "No printLevel() function for this qp" << std::endl; }
    virtual double SI_feasibilityTolerance() const { std::cout << "No feasibilityTolerance() function for this qp" << std::endl; return 0.; }
    virtual void SI_feasibilityTolerance(double) { std::cout << "No feasibilityTolerance(double) function for this qp" << std::endl; }
    virtual bool SI_warmStart() const { std::cout << "No warmStart() function for this qp" << std::endl; return false; }
    virtual void SI_warmStart(bool) { std::cout << "No warmStart(bool) function for this qp" << std::endl; }
    virtual const Eigen::VectorXd& SI_result() const = 0;
    virtual void SI_problem(int nrVar, int nrEq, int nrInEq) = 0;
    virtual bool SI_solve(const Eigen::MatrixXd& Q, const Eigen::VectorXd& c, const Eigen::MatrixXd& Aeq, const Eigen::VectorXd& beq,
        const Eigen::MatrixXd& Aineq, const Eigen::VectorXd& bineq, const Eigen::VectorXd& XL, const Eigen::VectorXd& XU) = 0;
};

// The new backend: batched Goldfarb-Idnani on the GPU, batch of one through the raw-QP entry.
// Fail codes and SI_iter have QuadProgDenseSolver's meaning (reference include/QuadProgSolver.h:21-27).
class B200Solver : public SolverInterface {
public:
    B200Solver() = default;
    int SI_fail() const override { return fail_; }
    int SI_iter() const override { return iter_[0]; }
    void SI_inform() const override
    {
        switch (fail_) {
        case 0: std::cout << "No problems" << std::endl; break;
        case 1: std::cout << "The minimization problem has no solution" << std::endl; break;
        case 2: std::cout << "Problems with the decomposition of Q (Is it symmetric?)" << std::endl; break;
        default: std::cout << "B200Solver: iteration limit reached" << std::endl; break;
        }
    }
    const Eigen::VectorXd& SI_result() const override { return result_; }
    void SI_problem(int nrVar, int nrEq, int nrInEq) override
    {
        nrVar_ = nrVar; nrEq_ = nrEq; nrInEq_ = nrInEq;
        result_.resize(nrVar);
        iact_.assign(size_t(nrVar), 0);
    }
    bool SI_solve(const Eigen::MatrixXd& Q, const Eigen::VectorXd& c, const Eigen::MatrixXd& Aeq, const Eigen::VectorXd& beq,
        const Eigen::MatrixXd& Aineq, const Eigen::VectorXd& bineq, const Eigen::VectorXd& XL, const Eigen::VectorXd& XU) override
    {
        const int n = int(c.rows()), meq = int(beq.rows()), m = int(bineq.rows());
        if (n != nrVar_) SI_problem(n, meq, m);
        b200::check(copra_b200_solve_qp_batch(b200::handle(), n, meq, m, 1, b200::arr(Q.data()), b200::arr(c.data()),
            b200::arr(meq ? Aeq.data() : nullptr), b200::arr(meq ? beq.data() : nullptr), b200::arr(m ? Aineq.data() : nullptr),
            b200::arr(m ? bineq.data() : nullptr), b200::arr(XL.data()), b200::arr(XU.data()), result_.data(), &fail_, iter_, &nact_,
            iact_.data(), COPRA_B200_HOST));
        return fail_ == 0;
    }
    // active set of the last solve: 1-based indices in [eq | ineq | upper | lower] space, add order
    std::vector<int> activeSet() const { return std::vector<int>(iact_.begin(), iact_.begin() + nact_); }
    int drops() const { return iter_[1]; }
    // used by LMPC's fused path
    void adopt(const Eigen::VectorXd& x, int fail, const int iter[2], int nact, const std::vector<int>& iact)
    {
        result_ = x; fail_ = fail; iter_[0] = iter[0]; iter_[1] = iter[1]; nact_ = nact; iact_ = iact;
    }

private:
    Eigen::VectorXd result_;
    int nrVar_ = 0, nrEq_ = 0, nrInEq_ = 0, fail_ = 0, nact_ = 0;
    int iter_[2] = { 0, 0 };
    std::vector<int> iact_;
};

// DEFAULT first and QuadProgDense last as in the reference enum (include/solverUtils.h:34-50); both now
// resolve to the same Goldfarb-Idnani method, executed on the GPU.
enum class SolverFlag { DEFAULT, B200, QuadProgDense };

inline std::unique_ptr<SolverInterface> solverFactory(SolverFlag) { return std::unique_ptr<SolverInterface>(new B200Solver()); }
inline SolverInterface* pythonSolverFactory(SolverFlag) { return new B200Solver(); }

// ====================================================================================================
// LMPC
// ====================================================================================================
class LMPC {
public:
    explicit LMPC(SolverFlag sFlag = SolverFlag::DEFAULT) : ps_(nullptr), sol_(solverFactory(sFlag)) {}
    explicit LMPC(const std::shared_ptr<PreviewSystem>& ps, SolverFlag sFlag = SolverFlag::DEFAULT) : sol_(solverFactory(sFlag))
    {
        initializeController(ps);
    }
    LMPC(const LMPC&) = delete;
    LMPC(LMPC&&) = default;
    LMPC& operator=(const LMPC&) = delete;
    LMPC& operator=(LMPC&&) = default;
    virtual ~LMPC() = default;

    void selectQPSolver(SolverFlag flag) { sol_ = solverFactory(flag); }
    void useSolver(std::unique_ptr<SolverInterface>&& solver) { sol_ = std::move(solver); }
    virtual void initializeController(const std::shared_ptr<PreviewSystem>& ps)
    {
        if (ps_) snapshotIfStale();
        ps_ = ps;
        clearConstraintMatrices();
    }

    // LMPC::solve (src/LMPC.cpp:79-101): updateSystem -> makeQPForm -> SI_problem -> SI_solve -> updateResults.
    bool solve()
    {
        using clock = std::chrono::high_resolution_clock;
        const auto t0 = clock::now();
        if (!ps_->isUpdated) ps_->updateSystem(); // fills the public Phi/Psi/xi once, like :233-235
        b200::Description D;
        describe(D);
        copra_b200_handle* h = b200::handle();
        copra_b200_sizes sz{};
        b200::check(copra_b200_lmpc_sizes(h, D.finish(), &sz));
        constraints_.nrEqConstr = sz.meq;
        constraints_.nrIneqConstr = sz.mineq;
        // results go to temporaries and are committed only on success: the reference leaves control() / trajectory() at
        // their previous values when the solver fails (updateResults is skipped, src/LMPC.cpp:95-97)
        Eigen::VectorXd control(sz.nU), trajectory(sz.X);
        bool success = false;
        B200Solver* native = dynamic_cast<B200Solver*>(sol_.get());
        if (native) {
            // fused K1..K7 in one call; SI_problem / SI_solve semantics are reproduced on the solver object
            Eigen::VectorXd x(sz.nvar);
            int status = -1, iters[2] = { 0, 0 }, nact = 0;
            std::vector<int> iact(size_t(sz.nvar), 0);
            copra_b200_results R{};
            R.control = control.data(); R.trajectory = trajectory.data(); R.x = x.data(); R.status = &status; R.iters = iters;
            R.nact = &nact; R.iact = iact.data(); R.memory = COPRA_B200_HOST;
            native->SI_problem(sz.nvar, sz.meq, sz.mineq);
            b200::check(copra_b200_lmpc_run(h, D.finish(), &R));
            myEpoch_ = b200::newEpoch();
            native->adopt(x, status, iters, nact, iact);
            copra_b200_timing tm{};
            copra_b200_last_timing(h, &tm);
            solveTime_ = tm.solve_ms * 1e-3;
            success = status == 0;
            matricesStale_ = true;
        } else {
            // any other SolverInterface: K1..K4 on the GPU, the plug-in solves, K7 on the GPU
            b200::check(copra_b200_lmpc_build(h, D.finish()));
            myEpoch_ = b200::newEpoch();
            fetchMatrices(sz);
            sol_->SI_problem(sz.nvar, sz.meq, sz.mineq);
            const auto t1 = clock::now();
            success = sol_->SI_solve(Q_, c_, Aeq_, beq_, Aineq_, bineq_, lb_, ub_);
            solveTime_ = std::chrono::duration<double>(clock::now() - t1).count();
            if (success) b200::check(copra_b200_lmpc_results(h, sol_->SI_result().data(), control.data(), trajectory.data(), COPRA_B200_HOST));
        }
        if (success) {
            control_ = control;
            trajectory_ = trajectory;
        }
        lastSizes_ = sz;
        checkDeleteCostsAndConstraints();
        solveAndBuildTime_ = std::chrono::duration<double>(clock::now() - t0).count();
        return success;
    }

    void inform() const noexcept { sol_->SI_inform(); }
    double solveTime() const noexcept { return solveTime_; }
    double solveAndBuildTime() const noexcept { return solveAndBuildTime_; }

    void addCost(const std::shared_ptr<CostFunction>& costFun)
    {
        snapshotIfStale();
        costFun->initializeCost(*ps_);
        spCost_.emplace_back(costFun);
    }
    void addConstraint(const std::shared_ptr<Constraint>& constr)
    {
        snapshotIfStale();
        constr->initializeConstraint(*ps_);
        switch (constr->constraintType()) { // src/LMPC.cpp:173-197
        case ConstraintFlag::EqualityConstraint: constraints_.spEqConstr.emplace_back(std::static_pointer_cast<EqIneqConstraint>(constr)); break;
        case ConstraintFlag::InequalityConstraint: constraints_.spIneqConstr.emplace_back(std::static_pointer_cast<EqIneqConstraint>(constr)); break;
        case ConstraintFlag::BoundConstraint: constraints_.spBoundConstr.emplace_back(std::static_pointer_cast<ControlBoundConstraint>(constr)); break;
        default: return;
        }
        constraints_.spConstr.emplace_back(constr);
    }
    void clearCosts() noexcept { snapshotIfStale(); spCost_.clear(); }
    void clearConstraints() noexcept
    {
        snapshotIfStale();
        constraints_ = Constraints();
        clearConstraintMatrices();
    }
    void removeCost(const std::shared_ptr<CostFunction>& costFun)
    {
        snapshotIfStale();
        auto it = std::find(spCost_.begin(), spCost_.end(), costFun);
        if (it != spCost_.end()) spCost_.erase(it);
    }
    void removeConstraint(const std::shared_ptr<Constraint>& constr)
    {
        snapshotIfStale();
        auto drop = [&](auto& vec) {
            for (auto it = vec.begin(); it != vec.end(); ++it)
                if (it->get() == constr.get()) { vec.erase(it); return; }
        };
        drop(constraints_.spConstr);
        drop(constraints_.spEqConstr);
        drop(constraints_.spIneqConstr);
        drop(constraints_.spBoundConstr);
    }

    const Eigen::VectorXd& control() const noexcept { return control_; }
    const Eigen::VectorXd& trajectory() const noexcept { return trajectory_; }
    int nrEqConstr() const noexcept { return constraints_.nrEqConstr; }
    int nrIneqConstr() const noexcept { return constraints_.nrIneqConstr; }
    const Eigen::MatrixXd& Q() const { refresh(); return Q_; }
    const Eigen::VectorXd& c() const { refresh(); return c_; }
    const Eigen::MatrixXd& Aineq() const { refresh(); return Aineq_; }
    const Eigen::VectorXd& bineq() const { refresh(); return bineq_; }
    const Eigen::MatrixXd& Aeq() const { refresh(); return Aeq_; }
    const Eigen::VectorXd& beq() const { refresh(); return beq_; }
    const Eigen::VectorXd& lb() const { refresh(); return lb_; }
    const Eigen::VectorXd& ub() const { refresh(); return ub_; }
    SolverInterface& solver() { return *sol_; }

protected:
    struct Constraints {
        int nrEqConstr = 0, nrIneqConstr = 0;
        std::vector<std::shared_ptr<Constraint>> spConstr;
        std::vector<std::shared_ptr<EqIneqConstraint>> spEqConstr, spIneqConstr;
        std::vector<std::shared_ptr<ControlBoundConstraint>> spBoundConstr;
    };

    virtual int nrVar() const { return ps_->fullUDim; }
    virtual void clearConstraintMatrices()
    {
        const int n = nrVar();
        Aineq_.resize(0, n); Aeq_.resize(0, n); bineq_.resize(0); beq_.resize(0);
        lb_ = Eigen::VectorXd::Constant(n, -std::numeric_limits<double>::max()); // :207-208 (quirk Q4)
        ub_ = Eigen::VectorXd::Constant(n, std::numeric_limits<double>::max());
    }
    // C-ABI description of this controller: costs in addCost order; equality, inequality and bound
    // constraints each in addConstraint order (the stacking order of src/LMPC.cpp:257-279).
    virtual void describe(b200::Description& D) const
    {
        D.system(*ps_);
        for (auto& c : spCost_) D.costs.push_back(c->describe());
        for (auto& c : constraints_.spConstr) D.cstrs.push_back(c->describe());
    }
    void fetchMatrices(const copra_b200_sizes& sz) const
    {
        b200::download(COPRA_B200_GET_Q, Q_, sz.nvar, sz.nvar);
        b200::download(COPRA_B200_GET_C, c_, sz.nvar);
        b200::download(COPRA_B200_GET_AEQ, Aeq_, sz.meq, sz.nvar);
        b200::download(COPRA_B200_GET_BEQ, beq_, sz.meq);
        b200::download(COPRA_B200_GET_AINEQ, Aineq_, sz.mineq, sz.nvar);
        b200::download(COPRA_B200_GET_BINEQ, bineq_, sz.mineq);
        b200::download(COPRA_B200_GET_LB, lb_, sz.nvar);
        b200::download(COPRA_B200_GET_UB, ub_, sz.nvar);
        matricesStale_ = false;
    }
    // The fused path leaves the assembled QP on the device; the getters pull it on demand.  If the
    // process-wide handle has built something else in the meantime, K1..K4 are re-run for this controller.
    // The getters must return the QP that was SOLVED (the reference fills Q_, c_, ... inside solve()): every call that
    // changes the description (add / remove / clear, the use_count purge, initializeController) first snapshots the
    // matrices through snapshotIfStale(), so a rebuild here always describes the solved problem; its sizes are re-queried
    // rather than trusted from the last solve.
    void refresh() const
    {
        if (!matricesStale_) return;
        copra_b200_sizes sz = lastSizes_;
        if (myEpoch_ != b200::buildEpoch()) {
            b200::Description D;
            describe(D);
            b200::check(copra_b200_lmpc_sizes(b200::handle(), D.finish(), &sz));
            b200::check(copra_b200_lmpc_build(b200::handle(), D.finish()));
            myEpoch_ = b200::newEpoch();
        }
        fetchMatrices(sz);
    }
    void snapshotIfStale() const noexcept
    {
        if (!matricesStale_) return;
        try { refresh(); } catch (...) { matricesStale_ = false; }
    }
    // use_count based auto-removal, after the solve (src/LMPC.cpp:288-307, quirk Q3)
    void checkDeleteCostsAndConstraints()
    {
        bool any = false;
        for (auto& c : constraints_.spConstr) any = any || c.use_count() <= 2;
        for (auto& c : spCost_) any = any || c.use_count() <= 1;
        if (any) snapshotIfStale(); // the getters keep returning the QP that was just solved
        auto purge = [](auto& sp, long limit, bool warn) {
            for (auto it = sp.begin(); it != sp.end();) {
                if (it->use_count() <= limit) {
                    if (warn) std::fprintf(stderr, "A '%s' has been destroyed.\nIt has been removed from the controller\n", (*it)->name().c_str());
                    it = sp.erase(it);
                } else ++it;
            }
        };
#ifdef NDEBUG
        const bool warn = false;
#else
        const bool warn = true;
#endif
        purge(constraints_.spConstr, 2, warn);
        purge(constraints_.spEqConstr, 2, false);
        purge(constraints_.spIneqConstr, 2, false);
        purge(constraints_.spBoundConstr, 2, false);
        purge(spCost_, 1, warn);
    }

    std::shared_ptr<PreviewSystem> ps_;
    std::unique_ptr<SolverInterface> sol_;
    std::vector<std::shared_ptr<CostFunction>> spCost_;
    Constraints constraints_;
    mutable Eigen::MatrixXd Q_, Aineq_, Aeq_;
    mutable Eigen::VectorXd c_, bineq_, beq_, lb_, ub_;
    Eigen::VectorXd control_, trajectory_;
    mutable bool matricesStale_ = false;
    mutable unsigned long myEpoch_ = 0;
    copra_b200_sizes lastSizes_{};
    double solveTime_ = 0, solveAndBuildTime_ = 0;
};

// ====================================================================================================
// InitialStateLMPC: decision vector [x0; U] (reference src/InitialStateLMPC.cpp)
// ====================================================================================================
class InitialStateLMPC : public LMPC {
public:
    explicit InitialStateLMPC(SolverFlag sFlag = SolverFlag::DEFAULT) : LMPC(sFlag) {}
    explicit InitialStateLMPC(const std::shared_ptr<PreviewSystem>& ps, SolverFlag sFlag = SolverFlag::DEFAULT)
        : LMPC(sFlag), R_(Eigen::MatrixXd::Zero(ps->xDim, ps->xDim)), r_(Eigen::VectorXd::Zero(ps->xDim)), x0lb_(ps->x0), x0ub_(ps->x0)
    {
        initializeController(ps);
    }
    Eigen::VectorXd initialState() const noexcept { return sol_->SI_result().head(ps_->xDim); }
    void resetInitialStateCost(const Eigen::MatrixXd& R, const Eigen::VectorXd& r) { R_ = R; r_ = r; }
    void resetInitialStateBounds(const Eigen::VectorXd& l, const Eigen::VectorXd& u) { x0lb_ = l; x0ub_ = u; }

protected:
    int nrVar() const override { return ps_->xDim + ps_->fullUDim; }
    void describe(b200::Description& D) const override
    {
        LMPC::describe(D);
        D.p.initial_state = 1;
        D.p.R = b200::arr(R_.data()); D.p.r = b200::arr(r_.data());
        D.p.x0lb = b200::arr(x0lb_.data()); D.p.x0ub = b200::arr(x0ub_.data());
    }
    Eigen::MatrixXd R_;
    Eigen::VectorXd r_, x0lb_, x0ub_;
};

// ====================================================================================================
// BatchedLMPC: the batched entry point -- `batch` controllers of one shape, solved in one call.
// Costs / constraints are added once as templates with per-instance parameter arrays: every array is a
// (pointer, stride) pair in column-major layout, stride 0 = shared by all instances.
// ====================================================================================================
class BatchedLMPC {
public:
    BatchedLMPC(int xDim, int uDim, int nrSteps, int batch, bool initialState = false, int memory = COPRA_B200_HOST)
    {
        if (nrSteps <= 0) COPRA_DOMAIN_ERROR("The number of step sould be a positive number! ");
        p_.nx = xDim; p_.nu = uDim; p_.N = nrSteps; p_.batch = batch; p_.initial_state = initialState ? 1 : 0; p_.memory = memory;
    }
    void system(copra_b200_array A, copra_b200_array B, copra_b200_array d, copra_b200_array x0) { p_.A = A; p_.B = B; p_.d = d; p_.x0 = x0; }
    void initialStateCost(copra_b200_array R, copra_b200_array r) { p_.R = R; p_.r = r; }
    void initialStateBounds(copra_b200_array lo, copra_b200_array up) { p_.x0lb = lo; p_.x0ub = up; }
    // full_size = COPRA_B200_PER_STEP: step-size matrices and a p / f / lower / upper with one vector per step (rows x steps
    // entries, step-major: the layout of AutoSpan::spanVector) -- references and limits that move over the horizon, on the
    // kernels of a step-size entry.  The descriptors are kept: retarget() re-reads the vectors they point to.
    int addCost(const copra_b200_cost& c) { costs_.push_back(c); return int(costs_.size()) - 1; }
    int addConstraint(const copra_b200_constraint& c) { cstrs_.push_back(c); return int(cstrs_.size()) - 1; }
    ~BatchedLMPC() { if (multi_) copra_b200_multi_destroy(multi_); }
    BatchedLMPC(const BatchedLMPC&) = delete;
    BatchedLMPC& operator=(const BatchedLMPC&) = delete;
    // Data-parallel sharding (SURVEY.md 8e): split the batch by instance index over these CUDA devices (one engine handle
    // and host thread per entry; an empty list = every visible device).  HOST arrays only.  Results are bitwise those of
    // a single-device solve.
    void useDevices(const std::vector<int>& devices)
    {
        if (p_.memory != COPRA_B200_HOST) COPRA_DOMAIN_ERROR("BatchedLMPC::useDevices takes HOST arrays (each shard is uploaded to its own device)");
        if (multi_) { copra_b200_multi_destroy(multi_); multi_ = nullptr; }
        const int rc = copra_b200_multi_create(devices.empty() ? nullptr : devices.data(), int(devices.size()), &multi_);
        if (rc) throw std::runtime_error("copra_b200_multi_create failed (no usable sm_100 CUDA device; there is no CPU fallback)");
        copra_b200_multi_set_warm_start(multi_, warm_ ? 1 : 0);
    }
    int nrDevices() const { return multi_ ? copra_b200_multi_size(multi_) : 1; }
    // SolverInterface::SI_warmStart(bool) for the batched engine (include/SolverInterface.h:42-45): resolve() seeds every
    // instance with the active set of its previous solve.  Same optimum; fewer iterations when the active sets move little.
    void warmStart(bool w) { warm_ = w; if (multi_) copra_b200_multi_set_warm_start(multi_, w ? 1 : 0); }
    bool warmStart() const { return warm_; }
    copra_b200_sizes sizes()
    {
        copra_b200_sizes s{};
        b200::check(copra_b200_lmpc_sizes(b200::handle(), finish(), &s));
        return s;
    }
    // returns the number of instances with status 0
    int solve()
    {
        const auto t0 = std::chrono::high_resolution_clock::now();
        const copra_b200_sizes s = sizes();
        const size_t B = size_t(p_.batch);
        controls_.assign(B * s.nU, 0.0); trajectories_.assign(B * s.X, 0.0);
        status_.assign(B, -1); iterations_.assign(2 * B, 0); nact_.assign(B, 0); iact_.assign(B * s.nvar, 0);
        copra_b200_results R{};
        R.control = controls_.data(); R.trajectory = trajectories_.data(); R.status = status_.data(); R.iters = iterations_.data();
        R.nact = nact_.data(); R.iact = iact_.data(); R.memory = COPRA_B200_HOST;
        if (multi_) {
            if (copra_b200_multi_lmpc_run(multi_, finish(), &R)) throw std::runtime_error(copra_b200_multi_last_error(multi_));
            solveTime_ = 0.0;
            for (int g = 0; g < copra_b200_multi_size(multi_); ++g) { // slowest shard's K5+K6 time
                copra_b200_timing tm{};
                if (copra_b200_multi_timing(multi_, g, &tm, nullptr) == 0) solveTime_ = std::max(solveTime_, double(tm.solve_ms) * 1e-3);
            }
            multiBuilt_ = true;
            solveAndBuildTime_ = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
            return int(std::count(status_.begin(), status_.end(), 0));
        }
        copra_b200_set_warm_start(b200::handle(), warm_ ? 1 : 0);
        b200::check(copra_b200_lmpc_run(b200::handle(), finish(), &R));
        myEpoch_ = b200::newEpoch();
        copra_b200_timing tm{};
        copra_b200_last_timing(b200::handle(), &tm);
        solveTime_ = tm.solve_ms * 1e-3;
        solveAndBuildTime_ = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
        return int(std::count(status_.begin(), status_.end(), 0));
    }
    // Receding-horizon step (reference usage: PreviewSystem::xInit + solve with isUpdated still set): only the initial
    // states change; condensing, Q and the constraint matrices stay resident on the device.  LMPC mode only.
    int resolve(copra_b200_array x0)
    {
        if (multi_ && multiBuilt_ && !p_.initial_state && p_.batch <= 65535) {
            const auto t0 = std::chrono::high_resolution_clock::now();
            copra_b200_results R{};
            R.control = controls_.data(); R.trajectory = trajectories_.data(); R.status = status_.data(); R.iters = iterations_.data();
            R.nact = nact_.data(); R.iact = iact_.data(); R.memory = COPRA_B200_HOST;
            if (copra_b200_multi_lmpc_resolve(multi_, x0, &R)) throw std::runtime_error(copra_b200_multi_last_error(multi_));
            p_.x0 = x0;
            solveAndBuildTime_ = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
            return int(std::count(status_.begin(), status_.end(), 0));
        }
        if (multi_ || myEpoch_ != b200::buildEpoch() || p_.batch > 65535 || p_.initial_state) {
            // another controller used the process-wide engine since, the batch was processed in chunks (only the last chunk
            // is resident), or x0 is a decision variable: full rebuild
            p_.x0 = x0;
            return solve();
        }
        const auto t0 = std::chrono::high_resolution_clock::now();
        copra_b200_results R{};
        R.control = controls_.data(); R.trajectory = trajectories_.data(); R.status = status_.data(); R.iters = iterations_.data();
        R.nact = nact_.data(); R.iact = iact_.data(); R.memory = COPRA_B200_HOST;
        b200::check(copra_b200_lmpc_resolve(b200::handle(), x0, p_.memory, &R));
        p_.x0 = x0;
        copra_b200_timing tm{};
        copra_b200_last_timing(b200::handle(), &tm);
        solveTime_ = tm.solve_ms * 1e-3;
        solveAndBuildTime_ = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
        return int(std::count(status_.begin(), status_.end(), 0));
    }
    // Receding-horizon step with new references and limits: new initial states, and the vectors (p, f, lower / upper) the
    // cost and constraint descriptors point to are read again; the matrices of the resident build are reused
    // (copra_b200_lmpc_retarget).  Falls back to solve() where resolve() does, and for full-size entries (their vector terms
    // are part of the dense assembly).
    int retarget(copra_b200_array x0)
    {
        p_.x0 = x0;
        bool dense = false;
        for (const auto& c : costs_) dense |= c.full_size == 1;
        for (const auto& c : cstrs_) dense |= c.full_size == 1 && c.kind != COPRA_B200_CSTR_CONTROL_BOUND;
        if (dense || p_.initial_state || p_.batch > 65535 || (multi_ ? !multiBuilt_ : myEpoch_ != b200::buildEpoch())) return solve();
        const auto t0 = std::chrono::high_resolution_clock::now();
        copra_b200_results R{};
        R.control = controls_.data(); R.trajectory = trajectories_.data(); R.status = status_.data(); R.iters = iterations_.data();
        R.nact = nact_.data(); R.iact = iact_.data(); R.memory = COPRA_B200_HOST;
        if (multi_) {
            if (copra_b200_multi_lmpc_retarget(multi_, finish(), &R)) throw std::runtime_error(copra_b200_multi_last_error(multi_));
        } else {
            b200::check(copra_b200_lmpc_retarget(b200::handle(), finish(), &R));
            copra_b200_timing tm{};
            copra_b200_last_timing(b200::handle(), &tm);
            solveTime_ = tm.solve_ms * 1e-3;
        }
        solveAndBuildTime_ = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
        return int(std::count(status_.begin(), status_.end(), 0));
    }
    // Sensitivities of the last solve / resolve / retarget (copra_b200_lmpc_vjp): the vector-Jacobian product of the controls
    // (dcontrol: nU x batch) and trajectories (dtrajectory: X x batch; either may be null) with respect to x0 and every entry's
    // vectors, written where `out` points (HOST arrays, batch-major; null = not wanted).  std::domain_error for full-size
    // entries other than the control bound and in initial-state mode; std::runtime_error when another controller has built
    // on the shared engine since this one's last solve.
    void vjp(const double* dcontrol, const double* dtrajectory, const copra_b200_vjp_out& out)
    {
        vjpImpl(dcontrol, dtrajectory, out, nullptr, nullptr);
    }
    // The same product together with the gradients with respect to every cost's weights and matrices
    // (copra_b200_lmpc_vjp_costs): costs.w / .M / .N per cost, rows, rows x nx and rows x nu per instance (column-major),
    // batch-major HOST arrays; null = not wanted.  Errors as vjp, plus std::domain_error for an M of a ControlCost or an N
    // of a TrajectoryCost / TargetCost.
    void vjp(const double* dcontrol, const double* dtrajectory, const copra_b200_vjp_out& out, const copra_b200_vjp_cost_out& costs)
    {
        vjpImpl(dcontrol, dtrajectory, out, &costs, nullptr);
    }
    // The same products together with the gradients with respect to the dynamics and the row constraints' matrices
    // (copra_b200_lmpc_vjp_model): model.A / .B / .d, nx x nx, nx x nu and nx per instance, model.E / .G per constraint, rows x
    // nx and rows x nu per instance (column-major), batch-major HOST arrays; null = not wanted; `costs` may be null.  Errors
    // as vjp, plus std::domain_error for an E of a constraint without E (ControlConstraint, bounds) or a G of one without G
    // (TrajectoryConstraint, bounds).
    void vjp(const double* dcontrol, const double* dtrajectory, const copra_b200_vjp_out& out, const copra_b200_vjp_cost_out* costs,
        const copra_b200_vjp_model_out& model)
    {
        vjpImpl(dcontrol, dtrajectory, out, costs, &model);
    }
    // Forward-mode sensitivities of the last solve (copra_b200_lmpc_jvp): dU (nU x k per instance) and dtrajectory (X x k)
    // along the in.ndir tangent directions of x0 and every entry's vectors described by `in` (HOST arrays, batch-major; either
    // output may be null).  Errors as vjp, plus std::domain_error for in.ndir < 1.
    void jvp(const copra_b200_jvp_in& in, double* dcontrol, double* dtrajectory)
    {
        sensGuard("jvp", false);
        sensCheck(multi_ ? copra_b200_multi_lmpc_jvp(multi_, &in, dcontrol, dtrajectory)
                         : copra_b200_lmpc_jvp(b200::handle(), &in, COPRA_B200_HOST, dcontrol, dtrajectory));
    }
    // The local feedback gain of the last solve (copra_b200_lmpc_feedback_gain): Ku = dU[0 : nu*steps]/dx0 ((nu*steps) x nx
    // per instance) and Kx = dtrajectory[0 : nx*(steps+1)]/dx0 ((nx*(steps+1)) x nx), column-major, batch-major HOST arrays;
    // either may be null.  Errors as jvp, with std::domain_error for steps outside [1, N].
    void feedbackGain(int steps, double* Ku, double* Kx)
    {
        sensGuard("feedbackGain", false);
        sensCheck(multi_ ? copra_b200_multi_lmpc_feedback_gain(multi_, steps, Ku, Kx)
                         : copra_b200_lmpc_feedback_gain(b200::handle(), steps, Ku, Kx, COPRA_B200_HOST));
    }
    // Sensitivities of the last solve of an initial-state controller (copra_b200_lmpc_vjp_initial_state): the vector-Jacobian
    // product with respect to x0 (through the x0 bounds that default to it) and every entry's vectors (`out`), and to R, r,
    // x0lb and x0ub (`init`: nx x nx, nx, nx, nx per instance; null = not wanted), batch-major HOST arrays.
    // std::runtime_error on an LMPC-mode controller or when another controller has built on the engine since this solve;
    // std::domain_error for full-size entries other than the control bound and for a gradient of an R, r, x0lb or x0ub the
    // controller was not given.
    void initialStateVjp(const double* dcontrol, const double* dtrajectory, const copra_b200_vjp_out& out,
        const copra_b200_vjp_initial_out& init)
    {
        sensGuard("initialStateVjp", true);
        sensCheck(multi_ ? copra_b200_multi_lmpc_vjp_initial_state(multi_, dcontrol, dtrajectory, &out, &init)
                         : copra_b200_lmpc_vjp_initial_state(b200::handle(), dcontrol, dtrajectory, COPRA_B200_HOST, &out, &init));
    }
    // Forward mode of the same (copra_b200_lmpc_jvp_initial_state): dU (nU x k per instance) and dtrajectory (X x k) along the
    // in.ndir tangent directions of `in` and `init` (R: nx x nx x k, r / x0lb / x0ub: nx x k per instance; null = zero).
    // Errors as initialStateVjp, plus std::domain_error for in.ndir < 1.
    void initialStateJvp(const copra_b200_jvp_in& in, const copra_b200_jvp_initial_in& init, double* dcontrol, double* dtrajectory)
    {
        sensGuard("initialStateJvp", true);
        sensCheck(multi_ ? copra_b200_multi_lmpc_jvp_initial_state(multi_, &in, &init, dcontrol, dtrajectory)
                         : copra_b200_lmpc_jvp_initial_state(b200::handle(), &in, &init, COPRA_B200_HOST, dcontrol, dtrajectory));
    }
    const std::vector<double>& controls() const { return controls_; }         // nU x batch, column-major
    const std::vector<double>& trajectories() const { return trajectories_; } // X x batch
    const std::vector<int>& status() const { return status_; }
    const std::vector<int>& iterations() const { return iterations_; }         // 2 x batch
    const std::vector<int>& nrActive() const { return nact_; }
    const std::vector<int>& activeSets() const { return iact_; }               // nvar x batch, 0 padded
    double solveTime() const { return solveTime_; }
    double solveAndBuildTime() const { return solveAndBuildTime_; }

private:
    const copra_b200_problem* finish()
    {
        p_.ncost = int(costs_.size()); p_.costs = costs_.data();
        p_.ncstr = int(cstrs_.size()); p_.cstrs = cstrs_.data();
        return &p_;
    }
    // copra_b200_lmpc_vjp_model (one KKT solve for all of them); costs and model null is copra_b200_lmpc_vjp
    void vjpImpl(const double* dcontrol, const double* dtrajectory, const copra_b200_vjp_out& out, const copra_b200_vjp_cost_out* costs,
        const copra_b200_vjp_model_out* model)
    {
        sensGuard("vjp", false);
        sensCheck(multi_ ? copra_b200_multi_lmpc_vjp_model(multi_, dcontrol, dtrajectory, &out, costs, model)
                         : copra_b200_lmpc_vjp_model(b200::handle(), dcontrol, dtrajectory, COPRA_B200_HOST, &out, costs, model));
    }
    // What every sensitivity method checks before it calls the engine: an initial-state controller for the initialState*
    // methods (std::runtime_error), HOST arrays (std::domain_error), and this controller's solve still resident on the
    // engine (std::runtime_error: another controller may have built on the shared engine since)
    void sensGuard(const char* name, bool initial) const
    {
        if (initial && !p_.initial_state) throw std::runtime_error(std::string("BatchedLMPC::") + name + " needs an initial-state controller; use vjp / jvp");
        if (p_.memory != COPRA_B200_HOST) COPRA_DOMAIN_ERROR(std::string("BatchedLMPC::") + name + " takes HOST arrays");
        if (multi_ ? !multiBuilt_ : myEpoch_ != b200::buildEpoch())
            throw std::runtime_error(std::string("BatchedLMPC::") + name + ": no solve of this controller is resident on the engine");
    }
    // The engine's error of a sensitivity call: E_ARG and E_UNSUPPORTED (a request this build cannot serve) as
    // std::domain_error, any other failure as std::runtime_error
    void sensCheck(int rc) const
    {
        if (!rc) return;
        const char* msg = multi_ ? copra_b200_multi_last_error(multi_) : copra_b200_last_error(b200::handle());
        if (rc == COPRA_B200_E_UNSUPPORTED || rc == COPRA_B200_E_ARG) COPRA_DOMAIN_ERROR(msg);
        throw std::runtime_error(msg);
    }
    copra_b200_problem p_{};
    std::vector<copra_b200_cost> costs_;
    std::vector<copra_b200_constraint> cstrs_;
    std::vector<double> controls_, trajectories_;
    std::vector<int> status_, iterations_, nact_, iact_;
    double solveTime_ = 0, solveAndBuildTime_ = 0;
    unsigned long myEpoch_ = ~0ul;
    copra_b200_multi* multi_ = nullptr;
    bool multiBuilt_ = false;
    bool warm_ = false;
};

} // namespace copra
