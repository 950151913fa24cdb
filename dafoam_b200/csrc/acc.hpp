// Data accessor of the reverse-sweep math (rev_kernels.hpp).  The hand-derived adjoint of a cell (revACell / revBCell /
// revCCell) reads and writes every value through GAcc: the global SoA arrays of the mesh, state, forward record, reverse
// intermediates and product vector, indexed by the (rank-local) cell or face id.  GAcc is the only place that knows the
// layout of those arrays (component strides nC or nCtot, interleaved U); the arithmetic only names values.  Reference role:
// the CoDiPack tape evaluation inside DASolver::dRdWTMatVecMultFunction (DASolver.C:1364-1409).
#pragma once
#include "views.hpp"

namespace dab
{

struct GAcc
{
    MeshView m;
    StateView s;
    RecordView r;
    AdjView a;
    PsiView x;
    double *yU, *yP, *yN, *yPhi; // segments of the product vector (U | p | nuTilda | phi)

    // ---- topology
    DAB_HD int maxCF() const { return m.maxCF; }
    DAB_HD int nIF() const { return m.nIF; }
    DAB_HD FaceRef face(int c, int k) const { return faceOf(m, c, k); }
    template <int NF>
    DAB_HD void faceRow(int c, int* e, int* n) const
    {
        _Pragma("unroll") for (int k = 0; k < NF; k++)
        {
            e[k] = m.cellFaces[(size_t)k * m.nC + c];
            n[k] = m.cellNbr[(size_t)k * m.nC + c];
        }
    }
    DAB_HD bool ghost(int n) const { return n >= m.nC; } // cell owned by another rank (several GPUs)
    DAB_HD int patch(int f) const { return m.bPatch[f - m.nIF]; }
    // ---- face data
    DAB_HD void Sf(int f, double* v) const { v[0] = m.Sx[f]; v[1] = m.Sy[f]; v[2] = m.Sz[f]; }
    DAB_HD void kv(int f, double* v) const { v[0] = m.kx[f]; v[1] = m.ky[f]; v[2] = m.kz[f]; }
    DAB_HD void Cf(int f, double* v) const { v[0] = m.Cfx[f]; v[1] = m.Cfy[f]; v[2] = m.Cfz[f]; }
    DAB_HD double magSf(int f) const { return m.magSf[f]; }
    DAB_HD double w(int f) const { return m.w[f]; }
    DAB_HD double delta(int f) const { return m.delta[f]; }
    DAB_HD double phi(int f) const { return s.phi[f]; }
    DAB_HD double xphi(int f) const { return x.phi[f]; }
    // ---- cell data: mesh, state, input vector
    DAB_HD double V(int c) const { return m.V[c]; }
    DAB_HD double yWall(int c) const { return m.yWall[c]; }
    DAB_HD double C(int c, int j) const { return (j == 0 ? m.Cx : (j == 1 ? m.Cy : m.Cz))[c]; }
    DAB_HD double U(int c, int j) const { return s.U[3 * c + j]; }
    DAB_HD double p(int c) const { return s.p[c]; }
    DAB_HD double nt(int c) const { return s.nt[c]; }
    DAB_HD double xU(int c, int j) const { return x.U[3 * c + j]; }
    DAB_HD double xp(int c) const { return x.p[c]; }
    DAB_HD double xnt(int c) const { return x.nt[c]; }
    // ---- forward record
    DAB_HD double nut(int c) const { return r.nut[c]; }
    DAB_HD double gU(int c, int i) const { return r.gU[(size_t)i * m.nCtot + c]; }
    DAB_HD double gP(int c, int i) const { return r.gP[(size_t)i * m.nCtot + c]; }
    DAB_HD double gNt(int c, int i) const { return r.gNt[(size_t)i * m.nCtot + c]; }
    DAB_HD double rAU(int c) const { return r.rAU[c]; }
    DAB_HD double HbyA(int c, int j) const { return r.HbyA[(size_t)j * m.nCtot + c]; }
    DAB_HD double D0(int c) const { return r.D0[c]; }
    DAB_HD double flag(int c) const { return r.flag[c]; }
    // ---- reverse intermediates
    DAB_HD double mt(int c, int j) const { return a.mt[(size_t)j * m.nCtot + c]; }
    DAB_HD double Dn(int c) const { return a.Dn[c]; }
    DAB_HD double Udir(int c, int j) const { return a.Udir[(size_t)j * m.nC + c]; }
    DAB_HD double pdir(int c) const { return a.pdir[c]; }
    DAB_HD double gPb(int c, int i) const { return a.gPb[(size_t)i * m.nCtot + c]; }
    DAB_HD double gUb(int c, int i) const { return a.gUb[(size_t)i * m.nCtot + c]; }
    DAB_HD double gNtb(int c, int i) const { return a.gNtb[(size_t)i * m.nCtot + c]; }
    DAB_HD double nutb(int c) const { return a.nutb[c]; }
    DAB_HD double U2(int c, int j) const { return a.U2[(size_t)j * m.nC + c]; }
    DAB_HD double nt2(int c) const { return a.nt2[c]; }
    DAB_HD void setMt(int c, int j, double v) const { a.mt[(size_t)j * m.nCtot + c] = v; }
    DAB_HD void setDn(int c, double v) const { a.Dn[c] = v; }
    DAB_HD void setUdir(int c, int j, double v) const { a.Udir[(size_t)j * m.nC + c] = v; }
    DAB_HD void setPdir(int c, double v) const { a.pdir[c] = v; }
    DAB_HD void setGPb(int c, int i, double v) const { a.gPb[(size_t)i * m.nCtot + c] = v; }
    DAB_HD void setGUb(int c, int i, double v) const { a.gUb[(size_t)i * m.nCtot + c] = v; }
    DAB_HD void setGNtb(int c, int i, double v) const { a.gNtb[(size_t)i * m.nCtot + c] = v; }
    DAB_HD void setNutb(int c, double v) const { a.nutb[c] = v; }
    DAB_HD void setU2(int c, int j, double v) const { a.U2[(size_t)j * m.nC + c] = v; }
    DAB_HD void setNt2(int c, double v) const { a.nt2[c] = v; }
    // ---- product vector
    DAB_HD void setYU(int c, int j, double v) const { yU[3 * c + j] = v; }
    DAB_HD void setYP(int c, double v) const { yP[c] = v; }
    DAB_HD void setYN(int c, double v) const { yN[c] = v; }
    DAB_HD void setYPhi(int f, double v) const { yPhi[f] = v; }
    // ---- optional features: MRF zone, adjoint of the boundary reference values (patchVelocity input)
    DAB_HD bool mrfCell(int c) const { return m.mrfCell && m.mrfCell[c]; }
    DAB_HD bool bcRefOn(int pa) const { return a.bcRefb && ((a.bcMask >> pa) & 1u); }
    DAB_HD bool bcRefAny() const { return a.bcRefb != nullptr; }
    DAB_HD void setBcRef(int c, int j, double v) const { a.bcRefb[(size_t)j * m.nC + c] = v; }
    DAB_HD void addBcRef(int c, int j, double v) const { a.bcRefb[(size_t)j * m.nC + c] += v; }
};

} // namespace dab
