// Solver::solvePrimal -- SIMPLE iterations on the device (reference DASimpleFoam::solvePrimal,
// src/adjoint/DASolver/DASimpleFoam/DASimpleFoam.C:123-185; loop/exit rule DASolver::loop, DASolver.C:156-228;
// residual bookkeeping DAUtility::primalResidualControl, DAUtility.C:734-801; failure rule
// DASolver::checkPrimalFailure).  Linear solvers: Jacobi sweeps for the (relaxed, diagonally dominant) momentum and
// nuTilda equations, PCG + multicolour symmetric Gauss-Seidel for the pressure equation; residuals are OpenFOAM's
// normalised L1 residuals so that primalMinResTol keeps its meaning.
#pragma once

namespace dab
{

inline void Solver::primalSetup()
{
    Primal& P = primal;
    if (P.allocated) return;
    const size_t nC = hm.nC, nT = hm.nCtot, mcf = hm.maxCF;
    P.uOff.alloc(be, mcf * nC); P.uDiag.alloc(be, 3 * nC); P.uB.alloc(be, 3 * nC);
    P.pOff.alloc(be, mcf * nC); P.pDiag.alloc(be, nC); P.pB.alloc(be, nC);
    P.nOff.alloc(be, mcf * nC); P.nDiag.alloc(be, nC); P.nB.alloc(be, nC);
    P.Utmp.alloc(be, 3 * nT); P.pOld.alloc(be, nT); P.ntTmp.alloc(be, nT);
    P.red.alloc(be, 6 * nC); P.ones.alloc(be, nC);
    P.r.alloc(be, nC); P.z.alloc(be, nT); P.d.alloc(be, nT); P.q.alloc(be, nC);
    if (P.consistent)
    {
        P.rAt.alloc(be, nT); P.gPOld.alloc(be, 3 * nT);
    }
    if (par.comp)
    {
        P.eOff.alloc(be, mcf * nC); P.eDiag.alloc(be, nC); P.eB.alloc(be, nC); P.heTmp.alloc(be, nT);
    }
    be.launch((int)nC, FillConst{P.ones.p, 1.0});
    primalOps.init(be, &comm, 8); // sums are all-reduced over the ranks
    P.ops = &primalOps;
    // greedy distance-1 colouring of the cell graph (hexahedral structured numbering: 2 colours)
    std::vector<int32_t> colourOf(nC, -1);
    int nCol = 0;
    {
        std::vector<int> mark;
        for (size_t c = 0; c < nC; c++)
        {
            mark.assign(nCol + 1, 0);
            for (size_t k = 0; k < mcf; k++)
            {
                const int n = hm.cellNbr[k * nC + c];
                if (n >= 0 && n < (int)nC && colourOf[n] >= 0) mark[colourOf[n]] = 1;
            }
            int col = 0;
            while (col < nCol && mark[col]) col++;
            if (col == nCol) nCol++;
            colourOf[c] = col;
        }
    }
    std::vector<int32_t> list(nC);
    P.colourStart.assign(nCol + 1, 0);
    for (size_t c = 0; c < nC; c++) P.colourStart[colourOf[c] + 1]++;
    for (int k = 0; k < nCol; k++) P.colourStart[k + 1] += P.colourStart[k];
    {
        std::vector<int> pos(P.colourStart.begin(), P.colourStart.end() - 1);
        for (size_t c = 0; c < nC; c++) list[pos[colourOf[c]]++] = (int32_t)c;
    }
    P.dColourOf.upload(be, colourOf);
    P.dColourList.upload(be, list);
    P.dS.alloc(be, 8);
    primalCoarseSetup();
    P.allocated = true;
}

// sums of the rows of P.red ([k][nC]) -> host
inline const double* Solver::primalSums(int k) { return primal.ops->dots(primal.red.p, hm.nC, k, primal.ones.p, hm.nC); }

// OpenFOAM normalised residual of a segregated equation at the current x; res[j] per component
inline void Solver::primalResidual(const EqnView& e, const double* x, const double* g, double* res)
{
    const int nC = hm.nC;
    const double nG = ghosted() ? (double)part.nGlobalCells : (double)nC;
    if (ghosted()) halo.exchangeCells({{const_cast<double*>(x), e.nc, e.nc == 3 ? 3 : 1, e.nc == 3 ? 1 : hm.nCtot}});
    be.launch(nC, StridedCopy{x, e.nc, e.nc, nC, primal.red.p});
    const double* s = primalSums(e.nc);
    if (e.nc == 3)
    {
        EqnResidual<3> k{e, x, g, mv.V, hm.nCtot, {0, 0, 0}, primal.red.p};
        for (int j = 0; j < 3; j++) k.xRef[j] = s[j] / (double)nG;
        be.launch(nC, k);
    }
    else
    {
        EqnResidual<1> k{e, x, g, mv.V, hm.nCtot, {s[0] / (double)nG, 0, 0}, primal.red.p};
        be.launch(nC, k);
    }
    s = primalSums(2 * e.nc);
    for (int j = 0; j < e.nc; j++) res[j] = s[j] / (s[e.nc + j] + 1e-20);
}

// Jacobi sweeps in pairs (x -> tmp -> x); returns the initial residuals
inline void Solver::primalJacobi(const EqnView& e, double* x, double* tmp, const double* g, const SegControl& ctl, double* res0)
{
    const int nC = hm.nC;
    primalResidual(e, x, g, res0);
    double mx0 = 0.0;
    for (int j = 0; j < e.nc; j++) mx0 = std::max(mx0, res0[j]);
    if (mx0 < ctl.tol) return;
    double res[3];
    for (int it = 0; it < ctl.maxIter; it += 4)
    {
        for (int rep = 0; rep < 2; rep++)
        {
            // ghost copies of the iterate after every sweep (one exchange per sweep on several ranks)
            if (e.nc == 3)
            {
                be.launch(nC, JacobiSweep<3>{e, x, tmp, g, mv.V, hm.nCtot});
                if (ghosted()) halo.exchangeCells({{tmp, 3, 3, 1}});
                be.launch(nC, JacobiSweep<3>{e, tmp, x, g, mv.V, hm.nCtot});
                if (ghosted()) halo.exchangeCells({{x, 3, 3, 1}});
            }
            else
            {
                be.launch(nC, JacobiSweep<1>{e, x, tmp, g, mv.V, hm.nCtot});
                if (ghosted()) halo.exchangeCells({{tmp, 1, 1, hm.nCtot}});
                be.launch(nC, JacobiSweep<1>{e, tmp, x, g, mv.V, hm.nCtot});
                if (ghosted()) halo.exchangeCells({{x, 1, 1, hm.nCtot}});
            }
        }
        primalResidual(e, x, g, res);
        bool done = true;
        for (int j = 0; j < e.nc; j++)
            if (!(res[j] < ctl.tol || res[j] < ctl.relTol * res0[j])) done = false;
        if (done) break;
    }
}

// aggregates of the pressure coarse space: recursive coordinate bisection of the cell centres (compact boxes)
inline void Solver::primalCoarseSetup()
{
    Primal& P = primal;
    const int nC = hm.nC;
    if (P.nAgg < 0) P.nAgg = std::min(1024, nC / 64);
    if (P.nAgg < 2)
    {
        P.nAgg = 0;
        return;
    }
    std::vector<int> part;
    rcbPartition(hm, P.nAgg, part);
    std::vector<int32_t> aggOf(part.begin(), part.end()), cnt(P.nAgg + 1, 0), cells(nC);
    for (int c = 0; c < nC; c++) cnt[aggOf[c] + 1]++;
    for (int a = 0; a < P.nAgg; a++) cnt[a + 1] += cnt[a];
    {
        std::vector<int32_t> pos(cnt.begin(), cnt.end() - 1);
        for (int c = 0; c < nC; c++) cells[pos[aggOf[c]]++] = c;
    }
    std::vector<int32_t> chunkStart, aggChunkOff(1, 0);
    for (int a = 0; a < P.nAgg; a++)
    {
        for (int i = cnt[a]; i < cnt[a + 1]; i += 32) chunkStart.push_back(i);
        aggChunkOff.push_back((int32_t)chunkStart.size());
    }
    chunkStart.push_back(nC);
    P.nChunks = (int)chunkStart.size() - 1;
    P.dAggOf.upload(be, aggOf);
    P.dAggCells.upload(be, cells);
    P.dAggStart.upload(be, cnt);
    P.dChunkStart.upload(be, chunkStart);
    P.dAggChunkOff.upload(be, aggChunkOff);
    P.dAc.alloc(be, (size_t)P.nAgg * P.nAgg);
    P.dColk.alloc(be, P.nAgg);
    P.dRc.alloc(be, P.nAgg);
    P.dYc.alloc(be, P.nAgg);
    P.dPartial.alloc(be, P.nChunks + 1);
}

// Galerkin coarse operator of the current pressure matrix and its inverse (device, Gauss-Jordan)
inline void Solver::primalCoarseRefresh(const EqnView& e)
{
    Primal& P = primal;
    if (P.nAgg == 0) return;
    const int n = P.nAgg;
    be.zero(P.dAc.p, (size_t)n * n * sizeof(double));
    be.launch(n, CoarseGalerkin{e, P.dAggOf.p, P.dAggCells.p, P.dAggStart.p, n, P.dAc.p});
    for (int k = 0; k < n; k++)
    {
        be.launch(n, GjStep1{P.dAc.p, P.dColk.p, n, k});
        be.launch(n * n, GjStep2{P.dAc.p, P.dColk.p, n, k});
    }
    P.coarseValid = true;
}

// z = M^{-1} r: multicolour symmetric Gauss-Seidel, M = (D+L) D^{-1} (D+U), plus the additive coarse correction
inline void Solver::primalPrecond(const EqnView& e, const double* r, double* z)
{
    const Primal& P = primal;
    const int nCol = (int)P.colourStart.size() - 1;
    for (int k = 0; k < nCol; k++)
        be.launch(P.colourStart[k + 1] - P.colourStart[k],
                  SgsColour{e, P.dColourList.p + P.colourStart[k], P.dColourOf.p, k, 0, r, z});
    for (int k = nCol - 2; k >= 0; k--)
        be.launch(P.colourStart[k + 1] - P.colourStart[k],
                  SgsColour{e, P.dColourList.p + P.colourStart[k], P.dColourOf.p, k, 1, r, z});
    if (P.nAgg > 0 && P.coarseValid)
    {
        be.launch(P.nChunks, CoarseRestrict1{r, P.dAggCells.p, P.dChunkStart.p, P.dPartial.p});
        be.launch(P.nAgg, CoarseRestrict2{P.dPartial.p, P.dAggChunkOff.p, P.dRc.p});
        be.launch(P.nAgg, CoarseApply{P.dAc.p, P.dRc.p, P.nAgg, P.dYc.p});
        be.launch(hm.nC, CoarseProlongAdd{P.dYc.p, P.dAggOf.p, z});
    }
}

// PCG on the (sign-flipped, SPD) pressure equation with the scalars kept on the device; the host only looks at the
// residual every few iterations.  Returns the iteration count, res0 = initial (OpenFOAM-normalised) residual
inline int Solver::primalPcg(const EqnView& e, double* x, const SegControl& ctl, double& res0)
{
    Primal& P = primal;
    const int nC = hm.nC;
    double r1[3];
    primalResidual(e, x, nullptr, r1);
    res0 = r1[0];
    if (res0 < ctl.tol) return 0;
    // norm factor once (OpenFOAM keeps it fixed during the solve)
    if (ghosted()) halo.exchangeCells({{x, 1, 1, hm.nCtot}});
    be.launch(nC, SpmvEll{e, x, P.q.p});
    be.launch(nC, ResidualOf{e.b, P.q.p, P.r.p});
    be.launch(nC, PcgProducts{P.r.p, P.r.p, P.r.p, P.red.p, P.red.p + nC});
    const double sumAbs0 = primalSums(2)[1];
    const double normFactor = sumAbs0 / res0;
    double* S = P.dS.p;
    const int checkEvery = 4;
    int it = 0;
    while (it < ctl.maxIter)
    {
        primalPrecond(e, P.r.p, P.z.p);
        be.launch(nC, PcgProducts{P.r.p, P.z.p, P.r.p, P.red.p, nullptr});
        P.ops->dotsDev(P.red.p, nC, 1, P.ones.p, nC, S + 0);
        be.launch(1, PcgScalarBeta{S, it == 0 ? 1 : 0});
        be.launch(nC, PcgUpdate2{S, P.z.p, P.d.p});
        if (ghosted()) halo.exchangeCells({{P.d.p, 1, 1, hm.nCtot}});
        be.launch(nC, SpmvEllProd{e, P.d.p, P.q.p, P.red.p});
        P.ops->dotsDev(P.red.p, nC, 1, P.ones.p, nC, S + 2);
        be.launch(1, PcgScalarAlpha{S});
        be.launch(nC, PcgUpdate1{S, P.d.p, P.q.p, x, P.r.p, P.red.p});
        P.ops->dotsDev(P.red.p, nC, 1, P.ones.p, nC, S + 3);
        it++;
        if (it % checkEvery == 0 || it == ctl.maxIter)
        {
            double sumAbs;
            be.d2h(&sumAbs, S + 3, sizeof(double));
            const double res = sumAbs / normFactor;
            if (!(res == res)) throw Error("pressure solver diverged (NaN)");
            if (res < ctl.tol || res < ctl.relTol * res0) break;
        }
    }
    return it;
}

inline int Solver::solvePrimal(PrimalStats& st)
{
    if (par.transonic)
        throw Error("solvePrimal: the transonic pressure corrector (pEqnRhoSimpleC.H / pEqnTurbo.H transonic branch, a non-symmetric "
                    "convection-diffusion pressure equation) is not built; the residual, its transpose product and the adjoint solve are");
    primalSetup();
    if (fvSourceDirty) updateFvSource();
    Primal& P = primal;
    const int nC = hm.nC, nT = hm.nCtot;
    auto t0 = std::chrono::steady_clock::now();
    EqnView eU{nC, hm.maxCF, 3, P.uOff.p, P.uDiag.p, P.uB.p, mv.cellNbr};
    EqnView eP{nC, hm.maxCF, 1, P.pOff.p, P.pDiag.p, P.pB.p, mv.cellNbr};
    EqnView eN{nC, hm.maxCF, 1, P.nOff.p, P.nDiag.p, P.nB.p, mv.cellNbr};
    st = PrimalStats();
    double maxRes = 0.0;
    int it = 0;
    EqnView eE{nC, hm.maxCF, 1, P.eOff.p, P.eDiag.p, P.eB.p, mv.cellNbr};
    const bool mr = ghosted();
    auto exGrad = [&]() {
        if (!mr) return;
        std::vector<HaloItem> it{{rv.gU, 9, 1, nT}, {rv.gP, 3, 1, nT}};
        if (par.turb) it.push_back({rv.gNt, 3, 1, nT});
        if (par.comp) it.push_back({rv.gHe, 3, 1, nT});
        halo.exchangeCells(it);
    };
    if (mr) exchangeStates();
    Params pp = par; // the primal kernels see the stored, relaxed density
    if (par.comp)
    {
        launchNF<cFwdA>(nT, mv, par, sv, rv); // rho = psi*p of the initial state (ghost cells included)
        pp.rhoFrozen = 1;
    }
    for (it = 1; par.comp && it <= P.maxIters; it++)
    {
        // ---- DARhoSimpleFoam: UEqnRhoSimple.H, EEqnRhoSimple.H, pEqnRhoSimple.H, turbulence.correct()
        maxRes = -1e10;
        be.d2d(P.pOld.p, dP.p, (size_t)nT * sizeof(double));
        launchNF<cFwdA>(nT, mv, pp, sv, rv);
        exGrad();
        launchNF<cUEqnAssemble>(nC, mv, pp, sv, rv, eU);
        primalJacobi(eU, dU.p, P.Utmp.p, rv.gP, P.cU, st.resU);
        {
            double s3[3] = {st.resU[0], st.resU[1], st.resU[2]};
            std::sort(s3, s3 + 3);
            maxRes = std::max(maxRes, s3[1]);
        }
        // energy: solve for he, T from he (thermo.correct())
        launchNF<cFwdA>(nT, mv, pp, sv, rv);
        exGrad();
        launchNF<cEEqnAssemble>(nC, mv, pp, sv, rv, eE, P.alphaE);
        {
            double re[3];
            primalJacobi(eE, rv.he, P.heTmp.p, nullptr, P.cE, re);
            st.resE = re[0];
            maxRes = std::max(maxRes, re[0]);
            be.launch(nC, TFromHe{pp, rv.he, dT.p});
            be.launch(nC, BoundField{dT.p, P.TMin, P.TMax}); // DAUtility::boundVar
            if (mr) halo.exchangeCells({{dT.p, 1, 1, nT}});
        }
        // pressure corrector
        launchNF<cFwdA>(nT, mv, pp, sv, rv);
        exGrad();
        be.launch(nC, HbyAKernel{eU, sv, rv, mv.V, nT});
        if (mr) halo.exchangeCells({{rv.rAU, 1, 1, nT}, {rv.HbyA, 3, 1, nT}});
        Simplec sc;
        if (P.consistent)
        {
            be.launch(nC, RAtKernel{eU, rv.rAU, mv.V, P.rAt.p});
            if (mr) halo.exchangeCells({{P.rAt.p, 1, 1, nT}});
            be.d2d(P.gPOld.p, rv.gP, (size_t)3 * nT * sizeof(double));
            sc = Simplec{P.rAt.p, P.pOld.p, P.gPOld.p};
        }
        launchNF<cPEqnAssemble>(nC, mv, pp, sv, rv, eP, sc);
        if (it == 1 || (it - 1) % P.coarseRefresh == 0) primalCoarseRefresh(eP);
        {
            double rp;
            st.pIterations += primalPcg(eP, dP.p, P.cP, rp);
            st.resP = rp;
            maxRes = std::max(maxRes, rp);
        }
        if (mr) halo.exchangeCells({{dP.p, 1, 1, nT}});
        launchNF<cPhiUpdate>(nC, mv, pp, sv, rv, dPhi.p, sc);
        if (mr) halo.exchangeFaces({{dPhi.p, 1, 1, hm.nF}});
        be.launch(nC, RelaxField{dP.p, P.pOld.p, P.alphaP});
        be.launch(nC, BoundField{dP.p, P.pMin, P.pMax});
        be.launch(nC, RhoRelax{pp, sv, rv.rho, P.alphaRho});
        if (mr) halo.exchangeCells({{dP.p, 1, 1, nT}, {rv.rho, 1, 1, nT}});
        launchNF<cFwdA>(nT, mv, pp, sv, rv); // grad of the relaxed p, closures at the new (p, T)
        exGrad();
        be.launch(nC, UCorrect{rv, dU.p, nT, sc});
        be.launch(3 * nC, BoundField{dU.p, -P.UMax, P.UMax});
        if (mr) halo.exchangeCells({{dU.p, 3, 3, 1}});
        if (par.turb)
        {
            launchNF<cFwdA>(nT, mv, pp, sv, rv);
            exGrad();
            launchNF<cNutEqnAssemble>(nC, mv, pp, sv, rv, eN, P.alphaN);
            double rn[3];
            primalJacobi(eN, dNt.p, P.ntTmp.p, nullptr, P.cN, rn);
            st.resN = rn[0];
            maxRes = std::max(maxRes, rn[0]);
            be.launch(nC, BoundField{dNt.p, P.ntMin, P.ntMax});
            if (mr) halo.exchangeCells({{dNt.p, 1, 1, nT}});
        }
        if (printInfo && (it % P.printInterval == 0 || it == 1))
            fprintf(stderr, "[dab200] SIMPLE %5d  U %.3e %.3e %.3e  he %.3e  p %.3e  nuTilda %.3e\n", it, st.resU[0], st.resU[1], st.resU[2], st.resE,
                    st.resP, st.resN);
        if (!(maxRes == maxRes)) break;
        if (maxRes < P.minResTol && it > P.minIters) break;
    }
    for (it = par.comp ? it : 1; !par.comp && it <= P.maxIters; it++)
    {
        maxRes = -1e10;
        be.d2d(P.pOld.p, dP.p, (size_t)nT * sizeof(double)); // p.storePrevIter()
        // --- momentum predictor (UEqnSimple.H)
        launchNF<FwdA>(nT, mv, par, sv, rv);
        exGrad();
        launchNFF<UEqnAssemble>(nC, mv, par, sv, rv, eU);
        primalJacobi(eU, dU.p, P.Utmp.p, rv.gP, P.cU, st.resU);
        {
            double s3[3] = {st.resU[0], st.resU[1], st.resU[2]};
            std::sort(s3, s3 + 3);
            maxRes = std::max(maxRes, s3[1]); // the median component (primalResidualControl for vectors)
        }
        // --- pressure corrector (pEqnSimple.H)
        be.launch(nC, HbyAKernel{eU, sv, rv, mv.V, nT});
        if (mr) halo.exchangeCells({{rv.rAU, 1, 1, nT}, {rv.HbyA, 3, 1, nT}});
        Simplec sc;
        if (P.consistent)
        {
            be.launch(nC, RAtKernel{eU, rv.rAU, mv.V, P.rAt.p});
            if (mr) halo.exchangeCells({{P.rAt.p, 1, 1, nT}});
            be.d2d(P.gPOld.p, rv.gP, (size_t)3 * nT * sizeof(double));
            sc = Simplec{P.rAt.p, P.pOld.p, P.gPOld.p};
        }
        for (int no = 0; no <= P.nNonOrth; no++)
        {
            if (no > 0)
            {
                launchNF<FwdA>(nT, mv, par, sv, rv); // grad(p) of the latest p for the non-orthogonal correction
                exGrad();
            }
            launchNF<PEqnAssemble>(nC, mv, par, sv, rv, eP, sc);
            if (no == 0 && (it == 1 || (it - 1) % P.coarseRefresh == 0)) primalCoarseRefresh(eP);
            double rp;
            st.pIterations += primalPcg(eP, dP.p, P.cP, rp);
            if (no == 0) st.resP = rp;
            maxRes = std::max(maxRes, rp);
        }
        if (mr) halo.exchangeCells({{dP.p, 1, 1, nT}});
        launchNF<PhiUpdate>(nC, mv, par, sv, rv, dPhi.p, sc);
        if (mr) halo.exchangeFaces({{dPhi.p, 1, 1, hm.nF}}); // cut faces: the owner rank's flux
        be.launch(nC, RelaxField{dP.p, P.pOld.p, P.alphaP});
        if (mr) halo.exchangeCells({{dP.p, 1, 1, nT}});
        launchNF<FwdA>(nT, mv, par, sv, rv); // grad of the relaxed p
        exGrad();
        be.launch(nC, UCorrect{rv, dU.p, nT, sc});
        if (mr) halo.exchangeCells({{dU.p, 3, 3, 1}});
        // --- turbulence (DASpalartAllmaras::correct)
        if (par.turb)
        {
            launchNF<FwdA>(nT, mv, par, sv, rv);
            exGrad();
            launchNF<NutEqnAssemble>(nC, mv, par, sv, rv, eN, P.alphaN);
            double rn[3];
            primalJacobi(eN, dNt.p, P.ntTmp.p, nullptr, P.cN, rn);
            st.resN = rn[0];
            maxRes = std::max(maxRes, rn[0]);
            be.launch(nC, BoundField{dNt.p, P.ntMin, P.ntMax});
            if (mr) halo.exchangeCells({{dNt.p, 1, 1, nT}});
        }
        if (printInfo && (it % P.printInterval == 0 || it == 1))
            fprintf(stderr, "[dab200] SIMPLE %5d  U %.3e %.3e %.3e  p %.3e  nuTilda %.3e\n", it, st.resU[0], st.resU[1], st.resU[2], st.resP, st.resN);
        if (!(maxRes == maxRes)) break; // NaN
        if (maxRes < P.minResTol && it > P.minIters) break;
    }
    st.iterations = std::min(it, P.maxIters);
    st.maxRes = maxRes;
    st.converged = maxRes < P.minResTol ? 1 : 0;
    // mirror the new state into the external layout (getOFFields) and invalidate what depended on the old one
    {
        const size_t n = nC;
        hWMirrorValid = false; // the states changed on the device
        be.d2d(dWext.p, dU.p, 3 * n * sizeof(double));
        be.d2d(dWext.p + 3 * n, dP.p, n * sizeof(double));
        size_t off = 4 * n;
        if (par.comp)
        {
            be.d2d(dWext.p + off, dT.p, n * sizeof(double));
            off += n;
        }
        if (par.turb)
        {
            be.d2d(dWext.p + off, dNt.p, n * sizeof(double));
            off += n;
        }
        be.d2d(dWext.p + off, dPhi.p, (size_t)hm.nF * sizeof(double));
    }
    be.sync();
    recorded = false;
    kry.pcValid = false;
    st.sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    // DASolver::checkPrimalFailure: fail if the residual misses the tolerance by more than primalMinResTolDiff (or NaN)
    if (!(maxRes == maxRes)) return 1;
    return (maxRes / P.minResTol > P.minResTolDiff) ? 1 : 0;
}

} // namespace dab
