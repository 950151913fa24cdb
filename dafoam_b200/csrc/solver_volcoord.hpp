// Solver::volCoordProduct -- [dR/dx_v]^T psi and dF/dx_v for the `volCoord` input (mesh point coordinates), and
// updateMesh (reference DASolvers::updateOFMesh).  See geom_kernels.hpp for the method (coloured central differences
// over the points, geometry and R(W) re-evaluated on the device).
#pragma once

namespace dab
{

// geometry arrays of the (possibly moved) host mesh -> the existing device buffers
inline void Solver::uploadGeometry()
{
    auto put = [&](DevBuf<double>& d, const std::vector<double>& h) { be.h2d(d.p, h.data(), h.size() * sizeof(double)); };
    for (int k = 0; k < 3; k++)
    {
        put(dS[k], hm.Sf[k]);
        put(dK[k], hm.corr[k]);
        put(dCf[k], hm.Cf[k]);
        put(dC[k], hm.C[k]);
    }
    put(dMagSf, hm.magSf);
    put(dW, hm.w);
    put(dDelta, hm.delta);
    put(dV, hm.V);
    updateMrfFlux();
    recorded = false;
    kry.pcValid = false;
}

// new point coordinates (the wall distance stays frozen: meshWaveFrozen)
inline void Solver::updateMesh(const double* pts)
{
    if (ghosted()) throw Error("updateOFMesh runs on one GPU in this build");
    std::copy(pts, pts + hm.points.size(), hm.points.begin());
    hm.computeGeometry();
    uploadGeometry();
    fvSourceDirty = fvSpec.nDisk > 0;
    if (volc.ready) be.h2d(volc.dPts0.p, hm.points.data(), hm.points.size() * sizeof(double));
}

inline void Solver::volCoordSetup()
{
    VolCoord& Vc = volc;
    if (Vc.ready) return;
    if (ghosted()) throw Error("the volCoord input runs on one GPU in this build");
    const int nC = hm.nC, nF = hm.nF, nP = hm.nP;
    // cells around each point
    std::vector<int> pcOff(nP + 1, 0), pcList;
    {
        std::vector<std::pair<int, int>> pr;
        pr.reserve((size_t)hm.fLab.size() * 2);
        for (int f = 0; f < nF; f++)
            for (int q = hm.fOff[f]; q < hm.fOff[f + 1]; q++)
            {
                pr.emplace_back(hm.fLab[q], hm.own[f]);
                if (f < hm.nIF) pr.emplace_back(hm.fLab[q], hm.nei[f]);
            }
        std::sort(pr.begin(), pr.end());
        pr.erase(std::unique(pr.begin(), pr.end()), pr.end());
        for (auto& x : pr) pcOff[x.first + 1]++;
        for (int p = 0; p < nP; p++) pcOff[p + 1] += pcOff[p];
        pcList.resize(pr.size());
        for (size_t i = 0; i < pr.size(); i++) pcList[i] = pr[i].second;
    }
    // home cell of every point: the surrounding cell that carries the fewest points so far
    std::vector<int> homed(nC, 0), homeOf(nP, -1), slotOf(nP, 0);
    for (int p = 0; p < nP; p++)
    {
        int best = -1;
        for (int i = pcOff[p]; i < pcOff[p + 1]; i++)
            if (best < 0 || homed[pcList[i]] < homed[best]) best = pcList[i];
        if (best < 0) continue; // unused point
        homeOf[p] = best;
        slotOf[p] = homed[best]++;
    }
    Vc.maxSlots = 1;
    for (int c = 0; c < nC; c++) Vc.maxSlots = std::max(Vc.maxSlots, homed[c]);
    std::vector<int32_t> slotPoint((size_t)nC * Vc.maxSlots, -1);
    for (int p = 0; p < nP; p++)
        if (homeOf[p] >= 0) slotPoint[(size_t)homeOf[p] * Vc.maxSlots + slotOf[p]] = p;
    // colour the home cells: two homes of one colour are more than 2*radius cells apart (disjoint footprints)
    detail::CellGraph G;
    G.build(hm);
    std::vector<int> colour(nC, -1);
    int nCol = 0;
    {
        std::vector<int> mark, ball;
        for (int c = 0; c < nC; c++)
        {
            if (homed[c] == 0) continue;
            G.ball(&c, 1, 2 * Vc.radius, ball);
            if ((int)mark.size() < nCol + 1) mark.resize(nCol + 1, -1);
            for (int x : ball)
                if (colour[x] >= 0) mark[colour[x]] = c;
            int k = 0;
            while (k < nCol && mark[k] == c) k++;
            if (k == nCol)
            {
                nCol++;
                mark.push_back(-1);
            }
            colour[c] = k;
        }
    }
    Vc.nColours = nCol;
    Vc.homeStart.assign(nCol + 1, 0);
    for (int c = 0; c < nC; c++)
        if (colour[c] >= 0) Vc.homeStart[colour[c] + 1]++;
    for (int k = 0; k < nCol; k++) Vc.homeStart[k + 1] += Vc.homeStart[k];
    std::vector<int32_t> homes(Vc.homeStart[nCol]);
    {
        std::vector<int> pos(Vc.homeStart.begin(), Vc.homeStart.end() - 1);
        for (int c = 0; c < nC; c++)
            if (colour[c] >= 0) homes[pos[colour[c]]++] = c;
    }
    // point lists per (colour, slot)
    Vc.listStart.assign((size_t)nCol * Vc.maxSlots + 1, 0);
    std::vector<int32_t> lists;
    for (int k = 0; k < nCol; k++)
        for (int s = 0; s < Vc.maxSlots; s++)
        {
            for (int i = Vc.homeStart[k]; i < Vc.homeStart[k + 1]; i++)
            {
                const int p = slotPoint[(size_t)homes[i] * Vc.maxSlots + s];
                if (p >= 0) lists.push_back(p);
            }
            Vc.listStart[(size_t)k * Vc.maxSlots + s + 1] = (int)lists.size();
        }
    // step per point: relStep * shortest edge at the point
    std::vector<double> eps(nP, 0.0), minEdge(nP, 1e300);
    for (int f = 0; f < nF; f++)
    {
        const int n = hm.fOff[f + 1] - hm.fOff[f];
        for (int i = 0; i < n; i++)
        {
            const int a = hm.fLab[hm.fOff[f] + i], b = hm.fLab[hm.fOff[f] + (i + 1) % n];
            double d2 = 0.0;
            for (int k = 0; k < 3; k++) d2 += (hm.points[3 * a + k] - hm.points[3 * b + k]) * (hm.points[3 * a + k] - hm.points[3 * b + k]);
            const double d = std::sqrt(d2);
            minEdge[a] = std::min(minEdge[a], d);
            minEdge[b] = std::min(minEdge[b], d);
        }
    }
    for (int p = 0; p < nP; p++) eps[p] = minEdge[p] < 1e299 ? Vc.relStep * minEdge[p] : 0.0;
    Vc.dFOff.upload(be, hm.fOff);
    Vc.dFLab.upload(be, hm.fLab);
    Vc.dSlotPoint.upload(be, slotPoint);
    Vc.dHomes.upload(be, homes);
    Vc.dLists.upload(be, lists);
    Vc.dEps.upload(be, eps);
    Vc.dPts.upload(be, hm.points);
    Vc.dPts0.upload(be, hm.points);
    Vc.dLabelA.alloc(be, nC);
    Vc.dLabelB.alloc(be, nC);
    Vc.dR2.alloc(be, nDof());
    Vc.dOut.alloc(be, (size_t)3 * nP);
    Vc.dF1.alloc(be, hm.nBF + 1);
    Vc.dF2.alloc(be, hm.nBF + 1);
    Vc.ready = true;
    if (printInfo)
    {
        int nEval = 0;
        for (size_t i = 0; i + 1 < Vc.listStart.size(); i++)
            if (Vc.listStart[i + 1] > Vc.listStart[i]) nEval += 6;
        fprintf(stderr, "[dab200] volCoord: %d colours x %d slots, %d residual evaluations per product\n", Vc.nColours, Vc.maxSlots, nEval);
    }
}

// out[3*nP] = [dR/dx_v]^T psi (function == nullptr) or seed * dF/dx_v
inline void Solver::volCoordProduct(const double* psi, const FunctionDef* function, double seed, double* out)
{
    volCoordSetup();
    VolCoord& Vc = volc;
    const int nC = hm.nC, nP = hm.nP;
    GeomView gv;
    gv.nC = nC; gv.nF = hm.nF; gv.nIF = hm.nIF; gv.maxCF = hm.maxCF;
    gv.fOff = Vc.dFOff.p; gv.fLab = Vc.dFLab.p; gv.own = dOwn.p; gv.nei = dNei.p; gv.cellFaces = dCellFaces.p;
    gv.pts = Vc.dPts.p;
    gv.Sx = dS[0].p; gv.Sy = dS[1].p; gv.Sz = dS[2].p; gv.magSf = dMagSf.p; gv.w = dW.p; gv.delta = dDelta.p;
    gv.kx = dK[0].p; gv.ky = dK[1].p; gv.kz = dK[2].p; gv.Cfx = dCf[0].p; gv.Cfy = dCf[1].p; gv.Cfz = dCf[2].p;
    gv.Cx = dC[0].p; gv.Cy = dC[1].p; gv.Cz = dC[2].p; gv.V = dV.p;
    auto geometry = [&]() {
        be.launch(hm.nF, GeomFaceK{gv});
        be.launch(nC, GeomCellK{gv});
        be.launch(hm.nF, GeomDerivedK{gv});
        if (fvSpec.nDisk > 0) be.launch(nC, FvSourceK{fvSpec, mv.Cx, mv.Cy, mv.Cz, nC, dFvS.p}); // the source follows the cell centres
        updateMrfFlux();                                                                           // and the relative fluxes the faces
    };
    if (psi) be.h2d(dX.p, psi, (size_t)nDof() * sizeof(double));
    be.d2d(Vc.dPts.p, Vc.dPts0.p, (size_t)3 * nP * sizeof(double));
    be.zero(Vc.dOut.p, (size_t)3 * nP * sizeof(double));
    const int ns = nCellStates(), offPhi = ns * nC;
    std::vector<ForceSpec> fsv;
    if (function)
    {
        ensureRecorded();
        fsv = derivativeSpecs(*function); // at the unperturbed geometry
    }
    auto evaluate = [&](double* Rdev, double* Fdev) {
        geometry();
        if (function)
        {
            if (par.comp)
            {
                launchNF<cFwdA>(hm.nCtot, mv, par, sv, rv);
                for (const ForceSpec& fs : fsv) be.launch(hm.nBF, cForceFwd{mv, par, sv, rv, fs, Fdev});
            }
            else
            {
                launchNF<FwdA>(hm.nCtot, mv, par, sv, rv);
                for (const ForceSpec& fs : fsv) be.launch(hm.nBF, ForceFwd{mv, par, sv, rv, fs, Fdev});
            }
        }
        else
            forward(0, Rdev, false);
    };
    for (int col = 0; col < Vc.nColours; col++)
    {
        // footprint labels of this colour's homes
        be.launch(nC, LabelInit{Vc.dLabelA.p});
        be.launch(Vc.homeStart[col + 1] - Vc.homeStart[col], LabelSeed{Vc.dLabelA.p, Vc.dHomes.p + Vc.homeStart[col]});
        int32_t *la = Vc.dLabelA.p, *lb = Vc.dLabelB.p;
        for (int r = 0; r < Vc.radius; r++)
        {
            be.launch(nC, LabelSweep{la, lb, mv.cellNbr, nC, hm.maxCF});
            std::swap(la, lb);
        }
        for (int slot = 0; slot < Vc.maxSlots; slot++)
        {
            const int l0 = Vc.listStart[(size_t)col * Vc.maxSlots + slot], l1 = Vc.listStart[(size_t)col * Vc.maxSlots + slot + 1];
            if (l1 == l0) continue;
            const int32_t* list = Vc.dLists.p + l0;
            for (int k = 0; k < 3; k++)
            {
                be.launch(l1 - l0, PointMove{Vc.dPts.p, Vc.dPts0.p, Vc.dEps.p, list, k, 1.0});
                evaluate(dR.p, Vc.dF1.p);
                be.launch(l1 - l0, PointMove{Vc.dPts.p, Vc.dPts0.p, Vc.dEps.p, list, k, -1.0});
                evaluate(Vc.dR2.p, Vc.dF2.p);
                be.launch(l1 - l0, PointMove{Vc.dPts.p, Vc.dPts0.p, Vc.dEps.p, list, k, 0.0});
                if (function)
                    be.launch(hm.nBF, VolCoordAccumF{mv, Vc.dF1.p, Vc.dF2.p, la, Vc.dSlotPoint.p, Vc.maxSlots, slot, k, Vc.dEps.p, seed, Vc.dOut.p});
                else
                    be.launch(nC, VolCoordAccumR{mv, ns, offPhi, dR.p, Vc.dR2.p, dX.p, la, Vc.dSlotPoint.p, Vc.maxSlots, slot, k,
                                                 Vc.dEps.p, Vc.dOut.p});
            }
        }
    }
    be.d2h(out, Vc.dOut.p, (size_t)3 * nP * sizeof(double));
    uploadGeometry(); // the unperturbed geometry exactly as the host computed it
    if (fvSpec.nDisk > 0) updateFvSource();
}

} // namespace dab
