// Hand-derived reverse sweep y = diag(n) (dR/dW)^T x of the forward kernels in fwd_kernels.hpp: the
// tape-free replacement of the reference's `globalADTape_.evaluate()` inside
// DASolver::dRdWTMatVecMultFunction (reference src/adjoint/DASolver/DASolver.C:1364-1409) followed by
// normalizeGradientVec (DASolver.C:2356-2455).
//
// The forward is cell <- faces <- cells gathers; its transpose is written as gathers too (each cell
// collects the adjoint contributions that the rows of its neighbours make to *its* variables), so the
// reverse needs no atomics and, on several GPUs, only plain ghost-cell copies between the stages.
//
//   RevA  adjoint of FwdC (pRes, phiRes -> HbyA, rAU, p, grad p) fused with the cell-level adjoint of
//         the momentum row (URes, rAU, HbyA -> m~ = Mbar/V, adjoint of the relaxed diagonal)
//   RevB  face-level adjoint of the momentum and SA rows: contributions of rows c and n to U_c, nuEff_c,
//         grad(U)_c, nuTilda_c, grad(nuTilda)_c and (owner side) phi_f
//   RevC  adjoint of FwdA (Gauss gradients, nut) + final assembly and state scaling
//
// Non-smooth intrinsics differentiate the active branch (max/min/fabs/upwind switches), sqrt has zero
// derivative at zero -- the same conventions as CoDiPack in the reference and as oracle/tape.hpp.
#pragma once
#include "views.hpp"
#include "acc.hpp"
#include "fwd_kernels.hpp"
#include <cmath>

namespace dab
{

DAB_HD double sgn(double x) { return x < 0.0 ? -1.0 : 1.0; }

// adjoint of saSource with seed z: accumulates into ntb, gUb[9], gNb[3]
DAB_HD void saSourceAdj(double nt, double nu, double y, const double* gU, const double* gN, double z, double& ntb, double* gUb, double* gNb, int fv3,
                        double* nub = nullptr) // nub: adjoint of the laminar viscosity (compressible: nu = mu(T)/rho)
{
    // every quotient below goes through a shared reciprocal (frcp: no IEEE-division slow path, views.hpp): 8 reciprocals instead of
    // 25 divisions per cell, and no conditional CALL between the loads of the kernel that inlines this
    const double inu = frcp(nu);
    const double chi = nt * inu;
    const double c3 = chi * chi * chi, den1 = c3 + SA::Cv1c, iden1 = frcp(den1);
    const double fv1 = c3 * iden1;
    const double den = 1.0 + chi * fv1, iden = frcp(den);
    const double fv2 = 1.0 - chi * iden;
    const double w01 = 0.5 * (gU[3] - gU[1]), w02 = 0.5 * (gU[6] - gU[2]), w12 = 0.5 * (gU[7] - gU[5]);
    const double Q = w01 * w01 + w02 * w02 + w12 * w12;
    const double sQ = sqrt(Q);
    const double Omega = 2.0 * sQ;
    const double ky2 = (SA::kappa * y) * (SA::kappa * y), iky2 = frcp(ky2), iy2 = iky2 * (SA::kappa * SA::kappa);
    // fv3 variant: St = f3*Omega + f2v*nt/ky2 (no clip)
    constexpr double iCv2 = 1.0 / SA::Cv2;
    const double t = 1.0 + chi * iCv2, t3 = t * t * t, c2 = chi * iCv2;
    const double it3 = fv3 ? frcp(t3) : 0.0;
    const double f2v = it3;
    const double Bq = (3.0 * t + c2 * c2) * it3;
    const double f3 = den * Bq * iCv2; // den = 1 + chi*fv1
    const double S1 = fv3 ? f3 * Omega + f2v * nt * iky2 : Omega + fv2 * nt * iky2, S2 = SA::Cs * Omega;
    const bool b1 = fv3 ? true : S1 > S2;
    const double St = b1 ? S1 : S2;
    const bool bS = St > 1e-15;
    const double Sm = bS ? St : 1e-15;
    const double iSmk = frcp(Sm * ky2);
    const double rr0 = nt * iSmk;
    const bool bR = rr0 < 10.0;
    const double rr = bR ? rr0 : 10.0;
    const double r2 = rr * rr, r5 = r2 * r2 * rr;
    const double g = rr + SA::Cw2 * (r5 * rr - rr);
    const double g2 = g * g, g6 = g2 * g2 * g2;
    const double ig6 = frcp(g6 + SA::Cw3p6);
    const double h = cbrt(sqrt((1.0 + SA::Cw3p6) * ig6)); // x^(1/6)
    const double fw = g * h;
    // reverse
    for (int i = 0; i < 3; i++) gNb[i] += -2.0 * (SA::Cb2 / SA::sigma) * gN[i] * z;
    double Stb = -SA::Cb1 * nt * z;
    ntb += (-SA::Cb1 * St + 2.0 * SA::Cw1 * fw * nt * iy2) * z;
    const double fwb = SA::Cw1 * nt * nt * iy2 * z;
    const double gb = fwb * h * SA::Cw3p6 * ig6;
    const double rrb = gb * (1.0 + SA::Cw2 * (6.0 * r5 - 1.0));
    const double rr0b = bR ? rrb : 0.0;
    ntb += rr0b * iSmk;
    const double Smb = -rr0b * nt * iSmk * frcp(Sm);
    if (bS) Stb += Smb;
    double Omegab = 0.0;
    if (fv3)
    {
        Omegab += f3 * Stb;
        ntb += Stb * f2v * iky2;
        // d f2v/d chi = -3 t^-4/Cv2;  d f3/d chi = [(fv1 + chi fv1') Bq + den dBq/dchi]/Cv2, dBq/dt = -(t^2 + 2t + 3)/t^4
        const double it4 = it3 * frcp(t);
        const double dfv1 = 3.0 * chi * chi * SA::Cv1c * iden1 * iden1;
        const double df2v = -3.0 * it4 * iCv2;
        const double dBq = -(t * t + 2.0 * t + 3.0) * it4 * iCv2;
        const double df3 = ((fv1 + chi * dfv1) * Bq + den * dBq) * iCv2;
        const double chib = Stb * (df3 * Omega + df2v * nt * iky2);
        ntb += chib * inu;
        if (nub) *nub -= chib * nt * inu * inu;
    }
    else if (b1)
    {
        Omegab += Stb;
        const double fv2b = Stb * nt * iky2;
        ntb += Stb * fv2 * iky2;
        double chib = -fv2b * iden * iden;
        const double fv1b = fv2b * chi * chi * iden * iden;
        chib += fv1b * 3.0 * chi * chi * SA::Cv1c * iden1 * iden1;
        ntb += chib * inu;
        if (nub) *nub -= chib * nt * inu * inu;
    }
    else
        Omegab += SA::Cs * Stb;
    if (sQ > 0.0)
    {
        const double Qb = Omegab * frcp(sQ);
        const double w01b = 2.0 * w01 * Qb, w02b = 2.0 * w02 * Qb, w12b = 2.0 * w12 * Qb;
        gUb[3] += 0.5 * w01b; gUb[1] -= 0.5 * w01b;
        gUb[6] += 0.5 * w02b; gUb[2] -= 0.5 * w02b;
        gUb[7] += 0.5 * w12b; gUb[5] -= 0.5 * w12b;
    }
}

// adjoint of the boundary gradient construction Gb[j*3+i] = gU[j*3+i] + nh_i (sng_j - sum_i nh_i gU[j*3+i])
DAB_HD void boundaryGradAdj(const double* nh, const double* Gbb, double* gUb, double* sngb)
{
    for (int j = 0; j < 3; j++)
    {
        const double t = nh[0] * Gbb[j * 3 + 0] + nh[1] * Gbb[j * 3 + 1] + nh[2] * Gbb[j * 3 + 2];
        sngb[j] += t;
        for (int i = 0; i < 3; i++) gUb[j * 3 + i] += Gbb[j * 3 + i] - nh[i] * t;
    }
}

// ---- face iteration through an accessor: hexahedral meshes (NF = 6) load the cell's whole row of the two tables before the face loop
// (all index loads in flight together; measured on B200: product 0.855 -> 0.763 ms), other meshes walk the ELL row
DAB_HD FaceRef faceOfE2(int nIF, int e, int n)
{
    FaceRef r;
    if (e < 0)
    {
        r.f = -1; r.n = -1; r.s = 0.0; r.bnd = false;
        return r;
    }
    r.f = e >> 1;
    r.s = (e & 1) ? -1.0 : 1.0;
    r.bnd = r.f >= nIF;
    r.n = n;
    return r;
}
#define DAB_ACC_FACES(NF)                                        \
    int e_[(NF) > 0 ? (NF) : 1], n_[(NF) > 0 ? (NF) : 1];        \
    if constexpr ((NF) > 0) A.faceRow<((NF) > 0 ? (NF) : 1)>(c, e_, n_);
#define DAB_ACC_FACE(NF, k) ((NF) > 0 ? faceOfE2(A.nIF(), e_[(NF) > 0 ? (k) : 0], n_[(NF) > 0 ? (k) : 0]) : A.face(c, k))

// RevA of one cell: adjoint of FwdC + cell-level adjoint of the momentum row
template <int NF>
DAB_HD void revACell(const GAcc& A, const Params& q, int c)
{
    const double Uc[3] = {A.U(c, 0), A.U(c, 1), A.U(c, 2)};
    const double V = A.V(c);
    const double rV = frcp(V);
    const double psiPc = A.xp(c) * (q.nrP ? rV : 1.0);
    double HbA[3] = {0, 0, 0}, rAUb = 0.0, pb = 0.0, gPb[3] = {0, 0, 0}, Ub[3] = {0, 0, 0};
    double refb[3] = {0, 0, 0};
    const double pc = A.p(c), rAUc = A.rAU(c);
    const double gPc[3] = {A.gP(c, 0), A.gP(c, 1), A.gP(c, 2)};
    DAB_ACC_FACES(NF)
    _Pragma("unroll") for (int k = 0; k < (NF > 0 ? NF : A.maxCF()); k++)
    {
        const FaceRef fr = DAB_ACC_FACE(NF, k);
        if (fr.f < 0) break;
        const int f = fr.f;
        // ---- load block: everything either branch reads, issued back to back with no control flow in between (a boundary face
        // "neighbour" is the cell itself: valid addresses, values unused).  The kernels are latency-bound; what limits them is
        // how many loads a thread has in flight, and a branch (or the slow-path CALL of an fp64 division) ends the region the
        // scheduler can batch loads in.
        const int n = fr.bnd ? c : fr.n;
        const double mS = A.magSf(f), dl = A.delta(f), xphif = A.xphi(f), w = A.w(f);
        double Sv[3], kv[3];
        A.Sf(f, Sv);
        A.kv(f, kv);
        const double xpn = A.xp(n), Vn = A.V(n), pn = A.p(n), rAUn = A.rAU(n);
        const double gPn[3] = {A.gP(n, 0), A.gP(n, 1), A.gP(n, 2)};
        const double rmS = frcp(mS);
        const double cphi = q.nrPhi ? rmS : 1.0;
        if (!fr.bnd)
        {
            const double psiPn = xpn * (q.nrP ? frcp(Vn) : 1.0);
            // F_f enters pRes_own with -1, pRes_nei with +1, phiRes_f with +1
            const double Fb = cphi * xphif - fr.s * (psiPc - psiPn);
            const double wc = fr.s > 0 ? w : 1.0 - w, wn = 1.0 - wc;
            double cg = 0.0;
            for (int j = 0; j < 3; j++) cg += kv[j] * (wc * gPc[j] + wn * gPn[j]);
            const double sn = fr.s * dl * (pn - pc) + cg; // delta*(p_N - p_P) + corr
            const double gam = wc * rAUc + wn * rAUn;
            for (int j = 0; j < 3; j++)
            {
                HbA[j] += wc * Sv[j] * Fb;
                gPb[j] -= gam * mS * wc * kv[j] * Fb;
            }
            rAUb -= wc * mS * sn * Fb;
            pb += fr.s * gam * mS * dl * Fb;
        }
        else
        {
            const int pa = A.patch(f);
            const double phib = A.phi(f);
            const double Fb = cphi * xphif - psiPc;
            const int kU = q.bcKind[F_U][pa];
            const bool assignable = (kU == BC_INLET_OUTLET || kU == BC_OUTLET_INLET || kU == BC_ZERO_GRADIENT);
            if (A.m.mrfType && A.m.mrfType[f - A.nIF()] == 1)
                ; // rotating wall of the MRF zone: the relative phiHbyA is identically zero
            else if (q.constrainHbyA && !assignable)
            {
                const double nh[3] = {Sv[0] * rmS, Sv[1] * rmS, Sv[2] * rmS};
                const double valb[3] = {Sv[0] * Fb, Sv[1] * Fb, Sv[2] * Fb};
                const double sngb[3] = {0.0, 0.0, 0.0};
                bcVectorAdj(kU, phib, dl, nh, valb, sngb, Ub);
                if (A.bcRefOn(pa)) bcVectorRefAdj(kU, phib, dl, valb, sngb, refb);
            }
            else
                for (int j = 0; j < 3; j++) HbA[j] += Sv[j] * Fb;
            double pv, sn, frp;
            bcScalar(q.bcKind[F_P][pa], q.bcVal[F_P][pa][0], pc, phib, dl, pv, sn, frp);
            rAUb -= mS * sn * Fb;
            const double snb = -rAUc * mS * Fb;
            pb -= frp * dl * snb;
        }
    }
    // cell-level adjoint of the momentum row: URes = cU*(M + grad p), HbyA = U - rAU*M, rAU = V/(Dn + icAvg)
    const double rAU = rAUc;
    const double rrAU = frcp(rAU);
    const double cU = q.nrU ? 1.0 : V;
    const double D0 = A.D0(c);
    double rAUtot = rAUb;
    double Mbv[3], Ud[3];
    for (int j = 0; j < 3; j++)
    {
        const double M = (Uc[j] - A.HbyA(c, j)) * rrAU;
        const double psiU = cU * A.xU(c, j);
        const double Mb = psiU - rAU * HbA[j];
        Mbv[j] = Mb;
        rAUtot -= M * HbA[j];
        const double mt = Mb * rV;
        A.setMt(c, j, mt);
        Ud[j] = Ub[j] + HbA[j] + D0 * mt;
        A.setGPb(c, j, gPb[j] + psiU);
    }
    if (A.mrfCell(c))
    {
        // adjoint of the Coriolis term M += Omega x U: Ub += Mb x Omega
        const double* w = A.m.mrfOmega;
        Ud[0] += Mbv[1] * w[2] - Mbv[2] * w[1];
        Ud[1] += Mbv[2] * w[0] - Mbv[0] * w[2];
        Ud[2] += Mbv[0] * w[1] - Mbv[1] * w[0];
    }
    for (int j = 0; j < 3; j++) A.setUdir(c, j, Ud[j]);
    A.setDn(c, -rAU * rAU * rAUtot * rV);
    A.setPdir(c, pb);
    if (A.bcRefAny())
        for (int j = 0; j < 3; j++) A.setBcRef(c, j, refb[j]);
}

template <int NF>
struct RevA
{
    MeshView m;
    Params q;
    StateView s;
    RecordView r;
    AdjView a;
    PsiView x;
    DAB_HD void operator()(int c) const
    {
        const GAcc A{m, s, r, a, x, nullptr, nullptr, nullptr, nullptr};
        revACell<NF>(A, q, c);
    }
};

// RevB of one cell.  FEAT: bit 0 = linearUpwindV limiter compiled in, bit 1 = wall-function nut BC compiled in, bit 2 = adjoint of
// the boundary reference values (patchVelocity input) compiled in (the common configuration without them keeps its register
// budget).
template <int NF, int FEAT>
DAB_HD void revBCell(const GAcc& A, const Params& q, int c)
{
    const int schU = q.divU, schN = q.divNut;
    const double Uc[3] = {A.U(c, 0), A.U(c, 1), A.U(c, 2)};
    const double nutc = A.nut(c);
    const double nuEc = nutc + q.nu;
    double gUc[9], gNc[3];
    for (int i = 0; i < 9; i++) gUc[i] = A.gU(c, i);
    const double ntc = q.turb ? A.nt(c) : 0.0;
    const double rsig = 1.0 / SA::sigma, rAl = frcp(q.alphaU); // one division per cell instead of one per face
    const double Gc = (ntc + q.nu) * rsig;
    for (int i = 0; i < 3; i++) gNc[i] = q.turb ? A.gNt(c, i) : 0.0;
    const double trc = gUc[0] + gUc[4] + gUc[8];
    const double V = A.V(c);
    const double Cc[3] = {A.C(c, 0), A.C(c, 1), A.C(c, 2)};
    // cell-level adjoints of row c
    const double mtc[3] = {A.mt(c, 0), A.mt(c, 1), A.mt(c, 2)};
    const double Dnc = A.Dn(c), flc = A.flag(c);
    const double D2c = Dnc * rAl;
    const double D1c = flc != 0.0 ? flc * D2c : 0.0;
    const double soc = flc != 0.0 ? 0.0 : D2c;
    const double D0c = D1c + mtc[0] * Uc[0] + mtc[1] * Uc[1] + mtc[2] * Uc[2];
    const double psiN = q.turb ? A.xnt(c) : 0.0;
    const double qc = psiN * (q.nrNut ? frcp(V) : 1.0); // adjoint of NV
    const double zc = psiN * (q.nrNut ? 1.0 : V);       // adjoint of the cell-local SA sources

    double U2[3] = {0, 0, 0}, nt2 = 0.0, nuEb = 0.0, gUb[9], gNb[3] = {0, 0, 0};
    double refb[3] = {0, 0, 0};
    for (int i = 0; i < 9; i++) gUb[i] = 0.0;

    DAB_ACC_FACES(NF)
    _Pragma("unroll") for (int k = 0; k < (NF > 0 ? NF : A.maxCF()); k++)
    {
        const FaceRef fr = DAB_ACC_FACE(NF, k);
        if (fr.f < 0) break;
        const int f = fr.f;
        // ---- load block (see revACell): the face's geometry and flux and the neighbour's record, issued with no control flow in
        // between; a boundary face reads the cell itself in place of a neighbour (valid addresses, values unused)
        const int n = fr.bnd ? c : fr.n;
        const double phi = A.phi(f), xphif = A.xphi(f);
        double Sv[3], kv[3], Cfv[3];
        A.Sf(f, Sv);
        A.kv(f, kv);
        A.Cf(f, Cfv);
        const double mS = A.magSf(f), dl = A.delta(f), wf = A.w(f);
        const double Un[3] = {A.U(n, 0), A.U(n, 1), A.U(n, 2)};
        const double nutn = A.nut(n), Dnn = A.Dn(n), fln = A.flag(n), Vn = A.V(n);
        const double mtn[3] = {A.mt(n, 0), A.mt(n, 1), A.mt(n, 2)};
        const double Cn[3] = {A.C(n, 0), A.C(n, 1), A.C(n, 2)};
        double gUn[9], gNn[3];
        for (int i = 0; i < 9; i++) gUn[i] = A.gU(n, i);
        const double ntn = q.turb ? A.nt(n) : 0.0, xntn = q.turb ? A.xnt(n) : 0.0;
        for (int i = 0; i < 3; i++) gNn[i] = q.turb ? A.gNt(n, i) : 0.0;
        const double mf = fr.s * phi;
        const double rmS = frcp(mS);
        double phib_acc = 0.0; // adjoint of phi_f (only meaningful on the owner side)
        if (!fr.bnd)
        {
            const double wc = fr.s > 0 ? wf : 1.0 - wf, wn = 1.0 - wc;
            const bool pos0 = phi >= 0.0;
            const double wupc = fr.s > 0 ? (pos0 ? 1.0 : 0.0) : (pos0 ? 0.0 : 1.0);
            const double nuEn = nutn + q.nu;
            const double D2n = Dnn * rAl;
            const double D1n = fln != 0.0 ? fln * D2n : 0.0;
            const double son = fln != 0.0 ? 0.0 : D2n;
            const double D0n = D1n + mtn[0] * Un[0] + mtn[1] * Un[1] + mtn[2] * Un[2];
            const bool ownUp = phi > 0.0;
            const bool cUp = fr.s > 0 ? ownUp : !ownUp;
            const double dC[3] = {Cfv[0] - Cc[0], Cfv[1] - Cc[1], Cfv[2] - Cc[2]};
            // ---- momentum rows c and n
            {
                const double wpc = schU == DIV_LINEAR ? wc : wupc;
                const double wpn = schU == DIV_LINEAR ? wn : 1.0 - wupc;
                const double gf = (wc * nuEc + wn * nuEn) * mS;
                const double g = gf * dl;
                const double offc = mf - wpc * mf - g;
                const double offn = -mf + wpn * mf - g;
                const double offbc = mtc[0] * Un[0] + mtc[1] * Un[1] + mtc[2] * Un[2] + sgn(offc) * soc;
                const double offbn = mtn[0] * Uc[0] + mtn[1] * Uc[1] + mtn[2] * Uc[2] + sgn(offn) * son;
                for (int j = 0; j < 3; j++) U2[j] += offn * mtn[j];
                const double abc = D0c - offbc, abn = D0n - offbn;
                double gb = abc + abn;   // adjoint of g
                double gfb = 0.0;        // adjoint of gf (non-orthogonal correction)
                const double lam[3] = {fr.s * (mtc[0] - mtn[0]), fr.s * (mtc[1] - mtn[1]), fr.s * (mtc[2] - mtn[2])};
                if (fr.s > 0)
                {
                    const double mbc = -D0c + offbc + wpc * abc;
                    const double mbn = -D0n + offbn + wpn * abn;
                    phib_acc += mbc - mbn;
                }
                if (!(FEAT & 1))
                {
                    // plain linearUpwind (compact form: no limiter state)
                    if (schU == DIV_LINEAR_UPWIND)
                    {
                        if (cUp)
                            for (int j = 0; j < 3; j++)
                                for (int i = 0; i < 3; i++) gUb[j * 3 + i] += dC[i] * phi * lam[j];
                        if (fr.s > 0)
                        {
                            const double* gu = cUp ? gUc : gUn;
                            double d[3];
                            for (int i = 0; i < 3; i++) d[i] = cUp ? dC[i] : Cfv[i] - Cn[i];
                            for (int j = 0; j < 3; j++)
                                phib_acc += (d[0] * gu[j * 3 + 0] + d[1] * gu[j * 3 + 1] + d[2] * gu[j * 3 + 2]) * lam[j];
                        }
                    }
                }
                else if (schU == DIV_LINEAR_UPWIND || schU == DIV_LINEAR_UPWIND_V)
                {
                    const double* gu = cUp ? gUc : gUn;
                    double d[3];
                    for (int i = 0; i < 3; i++) d[i] = cUp ? dC[i] : Cfv[i] - Cn[i];
                    double corr[3], corrL[3], outb[3], corrb[3] = {0, 0, 0};
                    for (int j = 0; j < 3; j++)
                    {
                        corr[j] = d[0] * gu[j * 3 + 0] + d[1] * gu[j * 3 + 1] + d[2] * gu[j * 3 + 2];
                        outb[j] = phi * lam[j]; // adjoint of the (limited) correction: +phi*corr into own row, -phi*corr into nei row
                    }
                    if ((FEAT & 1) && schU == DIV_LINEAR_UPWIND_V)
                    {
                        const double cf = ownUp ? (1.0 - wf) : -wf;
                        double maxCorr[3], maxCorrb[3] = {0, 0, 0};
                        for (int j = 0; j < 3; j++) maxCorr[j] = cf * fr.s * (Un[j] - Uc[j]);
                        luvLimit(corr, maxCorr, corrL);
                        luvLimitAdj(corr, maxCorr, outb, corrb, maxCorrb);
                        for (int j = 0; j < 3; j++) U2[j] -= cf * fr.s * maxCorrb[j];
                    }
                    else
                        for (int j = 0; j < 3; j++) { corrL[j] = corr[j]; corrb[j] = outb[j]; }
                    if (cUp)
                        for (int j = 0; j < 3; j++)
                            for (int i = 0; i < 3; i++) gUb[j * 3 + i] += dC[i] * corrb[j];
                    if (fr.s > 0)
                        for (int j = 0; j < 3; j++) phib_acc += corrL[j] * lam[j];
                }
                // non-orthogonal correction: MV_own -= gf*cg_j, MV_nei += gf*cg_j
                for (int j = 0; j < 3; j++)
                {
                    double cg = 0.0;
                    for (int i = 0; i < 3; i++) cg += kv[i] * (wc * gUc[j * 3 + i] + wn * gUn[j * 3 + i]);
                    gfb -= cg * lam[j];
                    const double cgb = -gf * lam[j];
                    for (int i = 0; i < 3; i++) gUb[j * 3 + i] += wc * kv[i] * cgb;
                }
                // dev2 term: MV_own -= fl_j, MV_nei += fl_j, fl = wc*tc + wn*tn
                double trb = 0.0;
                for (int j = 0; j < 3; j++)
                {
                    const double tcb = -wc * lam[j];
                    const double tcj = Sv[0] * gUc[0 * 3 + j] + Sv[1] * gUc[1 * 3 + j] + Sv[2] * gUc[2 * 3 + j] - (2.0 / 3.0) * trc * Sv[j];
                    nuEb += tcb * tcj;
                    for (int i = 0; i < 3; i++) gUb[i * 3 + j] += nuEc * Sv[i] * tcb;
                    trb -= (2.0 / 3.0) * nuEc * Sv[j] * tcb;
                }
                gUb[0] += trb; gUb[4] += trb; gUb[8] += trb;
                nuEb += wc * mS * (dl * gb + gfb);
            }
            // ---- SA rows c and n
            if (q.turb)
            {
                const double qn = xntn * (q.nrNut ? frcp(Vn) : 1.0);
                const double wpc = schN == DIV_LINEAR ? wc : wupc;
                const double wpn = schN == DIV_LINEAR ? wn : 1.0 - wupc;
                const double gf = (wc * Gc + wn * (ntn + q.nu) * rsig) * mS;
                const double g = gf * dl;
                nt2 += qc * (wpc * mf + g - mf) + qn * (-mf + wpn * mf - g);
                const double gb = (qc - qn) * (ntc - ntn);
                double gfb = 0.0;
                const double lam = fr.s * (qc - qn);
                if (fr.s > 0) phib_acc += qc * (1.0 - wpc) * (ntn - ntc) - qn * (1.0 - wpn) * (ntc - ntn);
                if (schN == DIV_LINEAR_UPWIND)
                {
                    if (cUp)
                        for (int i = 0; i < 3; i++) gNb[i] += dC[i] * phi * lam;
                    if (fr.s > 0)
                    {
                        double corr = 0.0;
                        for (int i = 0; i < 3; i++) corr += (cUp ? dC[i] * gNc[i] : (Cfv[i] - Cn[i]) * gNn[i]);
                        phib_acc += corr * lam;
                    }
                }
                double cg = 0.0;
                for (int i = 0; i < 3; i++) cg += kv[i] * (wc * gNc[i] + wn * gNn[i]);
                gfb -= cg * lam;
                const double cgb = -gf * lam;
                for (int i = 0; i < 3; i++) gNb[i] += wc * kv[i] * cgb;
                nt2 += wc * mS * (dl * gb + gfb) * rsig;
            }
        }
        else
        {
            const int pa = A.patch(f);
            const double nh[3] = {Sv[0] * rmS, Sv[1] * rmS, Sv[2] * rmS};
            const int kU = q.bcKind[F_U][pa];
            BCv bu;
            double uw[3];
            mrfWallRef(A.m, f, q.bcVal[F_U][pa], uw);
            bcVector(kU, uw, Uc, mf, dl, nh, bu);
            double ntb = 0.0, sngN = 0.0, frN = 0.0;
            if (q.turb) bcScalar(q.bcKind[F_NUTILDA][pa], q.bcVal[F_NUTILDA][pa][0], ntc, mf, dl, ntb, sngN, frN);
            double dP = 0.0, dNb = 0.0, dUn[3] = {0.0, 0.0, 0.0};
            double nutb = 0.0;
            if (q.turb)
                nutb = (FEAT & 2) ? nutBoundary<true>(q.bcKind[F_NUT][pa], q.bcVal[F_NUT][pa][0], nutc, ntb, q.nu, Uc, bu.val, dl, dP, dNb, dUn)
                                  : nutBoundaryBasic(q.bcKind[F_NUT][pa], q.bcVal[F_NUT][pa][0], nutc, ntb, q.nu, dP, dNb);
            const double nuEB = nutb + q.nu;
            const double G = nuEB * mS;
            // internalCoeffs and the argmax/argmin components used by relax()
            double ic[3];
            int kmax = 0, kmin = 0;
            for (int j = 0; j < 3; j++)
            {
                ic[j] = mf * bu.vic[j] - G * bu.gic[j];
                if (j > 0)
                {
                    if (fabs(ic[j]) > fabs(ic[kmax])) kmax = j;
                    if (ic[j] < ic[kmin]) kmin = j;
                }
            }
            double mb = -D0c, Gb_ = 0.0;
            for (int j = 0; j < 3; j++)
            {
                double icb = Dnc * (1.0 / 3.0);
                if (j == kmin) icb -= Dnc;
                if (j == kmax) icb += D1c * sgn(ic[j]);
                mb += bu.vic[j] * icb + mtc[j] * bu.val[j];
                Gb_ += -bu.gic[j] * icb - mtc[j] * bu.sng[j];
            }
            double valb[3], sngb[3];
            for (int j = 0; j < 3; j++) { valb[j] = mf * mtc[j]; sngb[j] = -G * mtc[j]; }
            // dev2 boundary term: MV_j -= nuEB * X_j
            double Gbd[9];
            for (int j = 0; j < 3; j++)
            {
                const double nG = nh[0] * gUc[j * 3 + 0] + nh[1] * gUc[j * 3 + 1] + nh[2] * gUc[j * 3 + 2];
                for (int i = 0; i < 3; i++) Gbd[j * 3 + i] = gUc[j * 3 + i] + nh[i] * (bu.sng[j] - nG);
            }
            const double trbv = Gbd[0] + Gbd[4] + Gbd[8];
            double nuEBb = mS * Gb_;
            double Gbb[9];
            for (int i = 0; i < 9; i++) Gbb[i] = 0.0;
            double trbb = 0.0;
            for (int j = 0; j < 3; j++)
            {
                const double X = Sv[0] * Gbd[0 * 3 + j] + Sv[1] * Gbd[1 * 3 + j] + Sv[2] * Gbd[2 * 3 + j] - (2.0 / 3.0) * trbv * Sv[j];
                nuEBb -= X * mtc[j];
                const double Xb = -nuEB * mtc[j];
                for (int i = 0; i < 3; i++) Gbb[i * 3 + j] += Sv[i] * Xb;
                trbb -= (2.0 / 3.0) * Sv[j] * Xb;
            }
            Gbb[0] += trbb; Gbb[4] += trbb; Gbb[8] += trbb;
            boundaryGradAdj(nh, Gbb, gUb, sngb);
            bcVectorAdj(kU, mf, dl, nh, valb, sngb, U2);
            if ((FEAT & 4) && A.bcRefOn(pa)) bcVectorRefAdj(kU, mf, dl, valb, sngb, refb);
            // nut_b -> nut_c / nuTilda_b / U_c (wall function)
            nuEb += dP * nuEBb;
            if (FEAT & 2)
                for (int j = 0; j < 3; j++) U2[j] += dUn[j] * nuEBb;
            double ntbb = dNb * nuEBb;
            if (q.turb)
            {
                const double Gs = (ntb + q.nu) * rsig * mS;
                mb += qc * (ntb - ntc);
                ntbb += qc * mf - qc * sngN * mS * rsig;
                const double sngNb = -qc * Gs;
                nt2 += -qc * mf + (1.0 - frN) * ntbb - frN * dl * sngNb;
            }
            phib_acc += mb;
        }
        if (fr.s > 0)
            A.setYPhi(f, (phib_acc - (q.nrPhi ? rmS : 1.0) * xphif) * phiRowScale(q, mS));
        else if (A.ghost(fr.n))
            A.setYPhi(f, 0.0); // cut face whose phi belongs to the neighbouring rank
    }
    if (q.turb) saSourceAdj(ntc, q.nu, A.yWall(c), gUc, gNc, zc, nt2, gUb, gNb, q.saFv3);
    for (int j = 0; j < 3; j++) A.setU2(c, j, U2[j]);
    if ((FEAT & 4) && A.bcRefAny())
        for (int j = 0; j < 3; j++) A.addBcRef(c, j, refb[j]);
    A.setNt2(c, nt2);
    A.setNutb(c, nuEb);
    for (int i = 0; i < 9; i++) A.setGUb(c, i, gUb[i]);
    for (int i = 0; i < 3; i++) A.setGNtb(c, i, gNb[i]);
}

template <int NF, int FEAT>
struct RevB
{
    MeshView m;
    Params q;
    StateView s;
    RecordView r;
    AdjView a;
    PsiView x;
    double* y;
    DAB_HD void operator()(int c) const
    {
        const GAcc A{m, s, r, a, x, nullptr, nullptr, nullptr, y + (size_t)(q.turb ? 5 : 4) * m.nC};
        revBCell<NF, FEAT>(A, q, c);
    }
};

// RevC of one cell: adjoint of FwdA (Gauss-gradient transpose, nut(nuTilda), BC adjoints) + final sum and state scaling
template <int NF>
DAB_HD void revCCell(const GAcc& A, const Params& q, int c, int functionMode)
{
    const double iVc = frcp(A.V(c));
    double Ub[3], pb = A.pdir(c), nb = 0.0;
    for (int j = 0; j < 3; j++) Ub[j] = A.Udir(c, j) + A.U2(c, j);
    double gUbc[9], gPbc[3], gNbc[3];
    for (int i = 0; i < 9; i++) gUbc[i] = A.gUb(c, i) * iVc;
    for (int i = 0; i < 3; i++)
    {
        gPbc[i] = A.gPb(c, i) * iVc;
        gNbc[i] = q.turb ? A.gNtb(c, i) * iVc : 0.0;
    }
    if (q.turb) nb = A.nt2(c) + A.nutb(c) * dnut_dnt(A.nt(c), q.nu);
    double refb[3] = {0, 0, 0};
    DAB_ACC_FACES(NF)
    _Pragma("unroll") for (int k = 0; k < (NF > 0 ? NF : A.maxCF()); k++)
    {
        const FaceRef fr = DAB_ACC_FACE(NF, k);
        if (fr.f < 0) break;
        const int f = fr.f;
        // load block (see revACell): the neighbour's gradient adjoints of an internal face, the cell's own for a boundary face
        const int n = fr.bnd ? c : fr.n;
        double Sv[3];
        A.Sf(f, Sv);
        const double wf = A.w(f), Vn = A.V(n);
        double gUbn[9], gPbn[3], gNbn[3];
        for (int i = 0; i < 9; i++) gUbn[i] = A.gUb(n, i);
        for (int i = 0; i < 3; i++)
        {
            gPbn[i] = A.gPb(n, i);
            gNbn[i] = q.turb ? A.gNtb(n, i) : 0.0;
        }
        const double So[3] = {fr.s * Sv[0], fr.s * Sv[1], fr.s * Sv[2]}; // outward
        if (!fr.bnd)
        {
            const double wc = fr.s > 0 ? wf : 1.0 - wf;
            const double iVn = frcp(Vn);
            for (int j = 0; j < 3; j++)
            {
                double t = 0.0;
                for (int i = 0; i < 3; i++) t += So[i] * (gUbc[j * 3 + i] - gUbn[j * 3 + i] * iVn);
                Ub[j] += wc * t;
            }
            double tp = 0.0, tn = 0.0;
            for (int i = 0; i < 3; i++)
            {
                tp += So[i] * (gPbc[i] - gPbn[i] * iVn);
                if (q.turb) tn += So[i] * (gNbc[i] - gNbn[i] * iVn);
            }
            pb += wc * tp;
            nb += wc * tn;
        }
        else
        {
            const int pa = A.patch(f);
            const double phib = A.phi(f), dl = A.delta(f);
            const double im = frcp(A.magSf(f));
            const double nh[3] = {Sv[0] * im, Sv[1] * im, Sv[2] * im};
            double valb[3];
            const double sngb[3] = {0.0, 0.0, 0.0};
            for (int j = 0; j < 3; j++) valb[j] = So[0] * gUbc[j * 3 + 0] + So[1] * gUbc[j * 3 + 1] + So[2] * gUbc[j * 3 + 2];
            bcVectorAdj(q.bcKind[F_U][pa], phib, dl, nh, valb, sngb, Ub);
            if (A.bcRefOn(pa)) bcVectorRefAdj(q.bcKind[F_U][pa], phib, dl, valb, sngb, refb);
            const double frp = bcFrac(q.bcKind[F_P][pa], phib);
            pb += (1.0 - frp) * (So[0] * gPbc[0] + So[1] * gPbc[1] + So[2] * gPbc[2]);
            if (q.turb)
            {
                const double frn = bcFrac(q.bcKind[F_NUTILDA][pa], phib);
                nb += (1.0 - frn) * (So[0] * gNbc[0] + So[1] * gNbc[1] + So[2] * gNbc[2]);
            }
        }
    }
    if (A.bcRefAny())
        for (int j = 0; j < 3; j++) A.addBcRef(c, j, refb[j]);
    for (int j = 0; j < 3; j++) A.setYU(c, j, Ub[j] * q.sU);
    A.setYP(c, pb * q.sP);
    if (q.turb) A.setYN(c, nb * q.sNut);
    if (functionMode)
    {
        // phi adjoint of a function: no face-flux dependence for the force function
        _Pragma("unroll") for (int k = 0; k < (NF > 0 ? NF : A.maxCF()); k++)
        {
            const FaceRef fr = DAB_ACC_FACE(NF, k);
            if (fr.f < 0) break;
            if (fr.s > 0 || A.ghost(fr.n)) A.setYPhi(fr.f, 0.0);
        }
    }
}

template <int NF>
struct RevC
{
    MeshView m;
    Params q;
    StateView s;
    RecordView r;
    AdjView a;
    double* y;
    int functionMode;
    DAB_HD void operator()(int c) const
    {
        const size_t nC = m.nC;
        const GAcc A{m, s, r, a, PsiView{}, y, y + 3 * nC, y + 4 * nC, y + (size_t)(q.turb ? 5 : 4) * nC};
        revCCell<NF>(A, q, c, functionMode);
    }
};

// ---- force function (DAFunctionForce.C:79-153) -------------------------------------------------------
struct ForceSpec
{
    unsigned mask; // bit p set: patch p contributes
    double dir[3]; // force direction, or the moment axis
    double scale;
    int mode;      // 0: force . dir (DAFunctionForce.C:79-153); 1: ((Cf - center) x force) . dir (DAFunctionMoment.C);
                   // 2: area-averaged total pressure p + 0.5 rho |U|^2 (DAFunctionTotalPressure.C); 3: mass flow rate rho U.Sf (DAFunctionMassFlowRate.C);
                   // 4 (compressible): area-averaged isentropic total pressure, one side of DAFunctionTotalPressureRatio.C
    double center[3];
    double areaSum;      // modes 2, 4: total area of the function's faces (all ranks)
    double gamma = 1.4;  // mode 4
    double shift = 0.0;  // modes 2, 4: subtracted from the face value before the area weighting; with shift = the average itself
                         // the geometric derivative of the area average needs no derivative of areaSum
    int accumulate = 0;  // ForceFwd: leave the faces outside the mask untouched (a second face group)
};

// boundary-face force contribution and (optionally) its adjoint w.r.t. the cell's variables
DAB_HD double forceFace(const MeshView& m, const Params& q, const StateView& s, const RecordView& r, const ForceSpec& fs, int f, int c,
                        double seed, double* Ub, double* pb, double* ntb_, double* nutPb, double* gUb)
{
    const int nT = m.nCtot;
    const int b = f - m.nIF, pa = m.bPatch[b];
    const double mS = m.magSf[f], dl = m.delta[f], phib = s.phi[f];
    const double Sv[3] = {m.Sx[f], m.Sy[f], m.Sz[f]};
    const double im = 1.0 / mS;
    const double nh[3] = {Sv[0] * im, Sv[1] * im, Sv[2] * im};
    const double Uc[3] = {s.U[3 * c], s.U[3 * c + 1], s.U[3 * c + 2]};
    double gUc[9];
    for (int i = 0; i < 9; i++) gUc[i] = r.gU[(size_t)i * nT + c];
    const int kU = q.bcKind[F_U][pa];
    BCv bu;
    double uw[3];
    mrfWallRef(m, f, q.bcVal[F_U][pa], uw);
    bcVector(kU, uw, Uc, phib, dl, nh, bu);
    double pv, snp, frp;
    bcScalar(q.bcKind[F_P][pa], q.bcVal[F_P][pa][0], s.p[c], phib, dl, pv, snp, frp);
    if (fs.mode >= 2)
    {
        // patch reductions of the boundary values (incompressible: rho = 1)
        const double U2 = bu.val[0] * bu.val[0] + bu.val[1] * bu.val[1] + bu.val[2] * bu.val[2];
        const double wA = mS / fs.areaSum;
        const double F = fs.scale * (fs.mode == 2 ? (pv + 0.5 * U2 - fs.shift) * wA : Sv[0] * bu.val[0] + Sv[1] * bu.val[1] + Sv[2] * bu.val[2]);
        if (gUb)
        {
            const double fb = seed * fs.scale;
            double valb[3];
            const double sngb[3] = {0.0, 0.0, 0.0};
            for (int j = 0; j < 3; j++) valb[j] = fs.mode == 2 ? fb * wA * bu.val[j] : fb * Sv[j];
            bcVectorAdj(kU, phib, dl, nh, valb, sngb, Ub);
            if (fs.mode == 2) *pb += (1.0 - frp) * fb * wA;
        }
        return F;
    }
    double ntb = 0.0, sngN = 0.0, frN = 0.0;
    const double ntc = q.turb ? s.nt[c] : 0.0;
    if (q.turb) bcScalar(q.bcKind[F_NUTILDA][pa], q.bcVal[F_NUTILDA][pa][0], ntc, phib, dl, ntb, sngN, frN);
    double dP = 0.0, dNb = 0.0, dUn[3] = {0.0, 0.0, 0.0};
    const double nutb = q.turb ? nutBoundary<true>(q.bcKind[F_NUT][pa], q.bcVal[F_NUT][pa][0], r.nut[c], ntb, q.nu, Uc, bu.val, dl, dP, dNb, dUn) : 0.0;
    const double nuEB = nutb + q.nu;
    double Gbd[9];
    for (int j = 0; j < 3; j++)
    {
        const double nG = nh[0] * gUc[j * 3 + 0] + nh[1] * gUc[j * 3 + 1] + nh[2] * gUc[j * 3 + 2];
        for (int i = 0; i < 3; i++) Gbd[j * 3 + i] = gUc[j * 3 + i] + nh[i] * (bu.sng[j] - nG);
    }
    const double trb = Gbd[0] + Gbd[4] + Gbd[8];
    // effective direction of this face: dir for a force, axis x r for a moment ((r x F).a = F.(a x r))
    double ed[3] = {fs.dir[0], fs.dir[1], fs.dir[2]};
    if (fs.mode == 1)
    {
        const double rv[3] = {m.Cfx[f] - fs.center[0], m.Cfy[f] - fs.center[1], m.Cfz[f] - fs.center[2]};
        ed[0] = fs.dir[1] * rv[2] - fs.dir[2] * rv[1];
        ed[1] = fs.dir[2] * rv[0] - fs.dir[0] * rv[2];
        ed[2] = fs.dir[0] * rv[1] - fs.dir[1] * rv[0];
    }
    double F = 0.0, sj[3];
    for (int j = 0; j < 3; j++)
    {
        // (Sf & dev(twoSymm(G)))_j = sum_i S_i (d_i U_j + d_j U_i) - 2/3 tr S_j
        double t = 0.0;
        for (int i = 0; i < 3; i++) t += Sv[i] * (Gbd[j * 3 + i] + Gbd[i * 3 + j]);
        sj[j] = t - (2.0 / 3.0) * trb * Sv[j];
        F += (Sv[j] * pv - nuEB * sj[j]) * ed[j];
    }
    F *= fs.scale;
    if (gUb)
    {
        double Gbb[9], sngb[3] = {0, 0, 0}, valb[3] = {0, 0, 0};
        for (int i = 0; i < 9; i++) Gbb[i] = 0.0;
        double pvb = 0.0, nuEBb = 0.0, trbb = 0.0;
        for (int j = 0; j < 3; j++)
        {
            const double fb = seed * fs.scale * ed[j];
            pvb += Sv[j] * fb;
            nuEBb -= sj[j] * fb;
            const double sb = -nuEB * fb;
            for (int i = 0; i < 3; i++)
            {
                Gbb[j * 3 + i] += Sv[i] * sb;
                Gbb[i * 3 + j] += Sv[i] * sb;
            }
            trbb -= (2.0 / 3.0) * Sv[j] * sb;
        }
        Gbb[0] += trbb; Gbb[4] += trbb; Gbb[8] += trbb;
        boundaryGradAdj(nh, Gbb, gUb, sngb);
        bcVectorAdj(kU, phib, dl, nh, valb, sngb, Ub);
        *pb += (1.0 - frp) * pvb;
        *nutPb += dP * nuEBb;
        *ntb_ += (1.0 - frN) * dNb * nuEBb;
        for (int j = 0; j < 3; j++) Ub[j] += dUn[j] * nuEBb;
    }
    return F;
}

struct ForceFwd
{
    MeshView m;
    Params q;
    StateView s;
    RecordView r;
    ForceSpec fs;
    double* out; // [nBF]
    DAB_HD void operator()(int b) const
    {
        const int f = m.nIF + b;
        const int pa = m.bPatch[b];
        if (!((fs.mask >> pa) & 1u))
        {
            if (!fs.accumulate) out[b] = 0.0;
            return;
        }
        out[b] = forceFace(m, q, s, r, fs, f, m.own[f], 0.0, nullptr, nullptr, nullptr, nullptr, nullptr);
    }
};

// seeds the reverse work arrays with dF/d(cell variables); RevC then propagates through the gradients
template <int NF>
struct ForceRevA
{
    MeshView m;
    Params q;
    StateView s;
    RecordView r;
    AdjView a;
    ForceSpec fs;
    double seed;
    DAB_HD void operator()(int c) const
    {
        const int nT = m.nCtot, nC = m.nC;
        double Ub[3] = {0, 0, 0}, pb = 0.0, ntb = 0.0, nutPb = 0.0, gUb[9];
        for (int i = 0; i < 9; i++) gUb[i] = 0.0;
        DAB_FACE_PREFETCH(NF)
        _Pragma("unroll") for (int k = 0; k < (NF > 0 ? NF : m.maxCF); k++)
        {
            const FaceRef fr = DAB_FACE(NF, k);
            if (fr.f < 0) break;
            if (!fr.bnd) continue;
            const int pa = m.bPatch[fr.f - m.nIF];
            if (!((fs.mask >> pa) & 1u)) continue;
            forceFace(m, q, s, r, fs, fr.f, c, seed, Ub, &pb, &ntb, &nutPb, gUb);
        }
        for (int j = 0; j < 3; j++)
        {
            a.Udir[(size_t)j * nC + c] = 0.0;
            a.U2[(size_t)j * nC + c] = Ub[j];
        }
        a.pdir[c] = pb;
        a.nt2[c] = ntb;
        a.nutb[c] = nutPb;
        for (int i = 0; i < 9; i++) a.gUb[(size_t)i * nT + c] = gUb[i];
    }
};

} // namespace dab
