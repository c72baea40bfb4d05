// active_rows.cuh -- the active constraint rows of a solved LMPC instance (LMPC mode, decision vector U), in their natural
// orientation: an Aeq / Aineq row read from the E A^k B tables with the indexing of K3's dev_fill_row (so the thin path never
// materialises Aineq), or e_k for either bound.  Shared by the sensitivity kernels K8 (k8_vjp.cu) and K9 (k9_jvp.cu).
#pragma once
#include "engine.cuh"

namespace cb {

// the family of general row `lrow` of Aeq (iseq) or Aineq, and its (step, line)
__device__ __forceinline__ int active_row_family(const BuildParams& P, bool iseq, int lrow, int& step, int& line)
{
    for (int k = 0; k < P.nfam; ++k) {
        const CstrFam& F = P.fam[k];
        if ((F.is_eq != 0) == iseq && lrow >= F.row_off && lrow < F.row_off + F.rows * (F.i1 - F.i0)) {
            step = F.i0 + (lrow - F.row_off) / F.rows;
            line = (lrow - F.row_off) % F.rows;
            return k;
        }
    }
    return -1;
}

// entry `col` of constraint `idx` (0-based in the solver's [eq | ineq | upper | lower] index space) of instance b;
// n = nU, nu = P.nu, mg = P.meq + P.mineq
__device__ __forceinline__ double active_row_entry(const BuildParams& P, int b, int n, int nu, int mg, int idx, int col)
{
    double v = 0.0;
    if (idx < mg) {
        const bool iseq = idx < P.meq;
        int i, l;
        const int fi = active_row_family(P, iseq, iseq ? idx : idx - P.meq, i, l);
        if (fi >= 0) {
            const CstrFam& F = P.fam[fi];
            const int j = col / nu, bb = col % nu, kk = i - j;
            if (kk >= 0) v = F.EGx[(long long)b * F.sEGx + l + F.rows * (bb + nu * kk)];
        }
    } else {
        const int var = (idx - mg) % n; // upper rows first, then lower rows
        v = (col == var) ? 1.0 : 0.0;
    }
    return v;
}

} // namespace cb
