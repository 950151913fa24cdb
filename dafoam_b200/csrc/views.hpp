// Device-side views (plain pointers, passed to kernels by value) and small inline helpers shared by
// the forward R(W) kernels and the hand-derived reverse kernels.
#pragma once
#include <cmath>
#include <cstdint>

#if defined(__CUDACC__)
#define DAB_HD __host__ __device__ __forceinline__
#else
#define DAB_HD inline
#endif

namespace dab
{

// Reciprocal without the slow-path branch of an IEEE fp64 division.  `a / b` compiles to MUFU.RCP64H + Newton steps + a
// conditional CALL for denormal / huge operands; that branch ends the scheduling region, so the loads of a face stay serialised
// behind it (the kernels are latency-bound: profiles/r02_latency_analysis.md).  For the operands it is used on (cell volumes,
// face areas: normal, positive) two Newton steps on rcp.approx give the correctly rounded result to within 1 ulp.
DAB_HD double frcp(double x)
{
#if defined(__CUDA_ARCH__)
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    return r;
#else
    return 1.0 / x;
#endif
}

constexpr int MAXP = 16; // max patches per rank
enum { F_U = 0, F_P = 1, F_NUTILDA = 2, F_NUT = 3, N_FIELDS = 4 };
enum { BC_FIXED_VALUE = 0, BC_ZERO_GRADIENT = 1, BC_INLET_OUTLET = 2, BC_OUTLET_INLET = 3, BC_SYMMETRY = 4, BC_CALCULATED = 5, BC_NUT_LOW_RE = 6, BC_NUT_SPALDING = 7 };
enum { DIV_UPWIND = 0, DIV_LINEAR_UPWIND = 1, DIV_LINEAR = 2, DIV_LINEAR_UPWIND_V = 3, DIV_LIMITED_LINEAR = 4 /* div(phid,p) only */ };

struct MeshView
{
    int nC, nCtot, nF, nIF, nBF, maxCF;
    const int32_t* own;       // [nF]
    const int32_t* nei;       // [nIF]
    const int32_t* cellFaces; // ELL [maxCF][nC]
    const int32_t* cellNbr;   // ELL [maxCF][nC]: the cell across face k (-1: boundary face or padding)
    const int32_t* bPatch;    // [nBF]
    const double *Sx, *Sy, *Sz, *magSf, *w, *delta, *kx, *ky, *kz, *Cfx, *Cfy, *Cfz; // [nF]
    const double *Cx, *Cy, *Cz, *V, *yWall;                                          // [nCtot]
    const double* fvS; // [3][nC] momentum source per unit volume (fvSource: actuator disks) or null
    // MRF zone (reference src/adjoint/DAMisc/MRFDF/MRFZoneDF.C) or null pointers: cell mask, boundary-face type
    // (MRFZoneDF::setMRFFaces: 1 included = rotating wall, 2 excluded), (Omega x (Cf - origin)) . Sf of the zone faces
    const unsigned char* mrfCell; // [nCtot]
    const unsigned char* mrfType; // [nBF]
    const double* mrfFlux;        // [nF], zero outside the zone
    double mrfOmega[3], mrfOrigin[3];
};

// reference value of the velocity boundary condition on boundary face f of patch value `patchVal`: the patch's own value, or the
// wall velocity Omega x (Cf - origin) on a rotating wall of the MRF zone (MRFZoneDF::correctBoundaryVelocity)
DAB_HD void mrfWallRef(const MeshView& m, int f, const double* patchVal, double* ref)
{
    ref[0] = patchVal[0];
    ref[1] = patchVal[1];
    ref[2] = patchVal[2];
    if (m.mrfType && m.mrfType[f - m.nIF] == 1)
    {
        const double r[3] = {m.Cfx[f] - m.mrfOrigin[0], m.Cfy[f] - m.mrfOrigin[1], m.Cfz[f] - m.mrfOrigin[2]};
        const double* w = m.mrfOmega;
        ref[0] = w[1] * r[2] - w[2] * r[1];
        ref[1] = w[2] * r[0] - w[0] * r[2];
        ref[2] = w[0] * r[1] - w[1] * r[0];
    }
}

// relative boundary flux (MRFZoneDF::makeRelativeRhoFlux): zero on a rotating wall, minus rho_b (Omega x r).Sf on an excluded face
DAB_HD double mrfBoundaryFlux(const MeshView& m, int f, double ph, double rhob)
{
    if (!m.mrfType) return ph;
    const int ty = m.mrfType[f - m.nIF];
    return ty == 1 ? 0.0 : (ty == 2 ? ph - rhob * m.mrfFlux[f] : ph);
}

// mrfFlux[f] = (Omega x (Cf - origin)) . Sf on the faces flagged in faceIn (internal faces touching the zone, excluded boundary
// faces of zone cells), zero elsewhere; recomputed whenever the geometry changes
struct MrfFluxK
{
    MeshView m;
    const unsigned char* faceIn;
    double* out;
    DAB_HD void operator()(int f) const
    {
        double v = 0.0;
        if (faceIn[f])
        {
            const double r[3] = {m.Cfx[f] - m.mrfOrigin[0], m.Cfy[f] - m.mrfOrigin[1], m.Cfz[f] - m.mrfOrigin[2]};
            const double* w = m.mrfOmega;
            v = (w[1] * r[2] - w[2] * r[1]) * m.Sx[f] + (w[2] * r[0] - w[0] * r[2]) * m.Sy[f] + (w[0] * r[1] - w[1] * r[0]) * m.Sz[f];
        }
        out[f] = v;
    }
};

// DAFvSourceActuatorDisk, source = cylinderAnnulusSmooth (reference src/adjoint/DAFvSource/DAFvSourceActuatorDisk.C:205-407):
// the 13 actuatorDiskPars (center, direction, innerRadius, outerRadius, scale, POD, expM, expN, targetThrust) + eps, rotDir
struct ActuatorDisk
{
    double par[13];
    double eps;
    int rotLeft;
};
constexpr int MAXDISK = 4;
struct FvSourceSpec
{
    int nDisk;
    ActuatorDisk disk[MAXDISK];
};

// source vector (force per unit volume) of one disk at the cell centre C
DAB_HD void actuatorDiskSource(const ActuatorDisk& d, const double* C, double* out)
{
    const double* a = d.par;
    const double dm = sqrt(a[3] * a[3] + a[4] * a[4] + a[5] * a[5]);
    const double dn[3] = {a[3] / dm, a[4] / dm, a[5] / dm};
    const double rin = a[6], rout = a[7], scale = a[8], POD = a[9], expM = a[10], expN = a[11], eps = d.eps;
    const double epsR = eps / (rout - rin), rMin = epsR, rMax = 1.0 - epsR;
    const double fRMin = pow(rMin, expM) * pow(1.0 - rMin, expN), fRMax = pow(rMax, expM) * pow(1.0 - rMax, expN);
    const double v[3] = {C[0] - a[0], C[1] - a[1], C[2] - a[2]};
    // "cellC2AVecE & dirNorm" with a diagonal tensor: the component-wise product (the reference's definition)
    const double vA[3] = {v[0] * dn[0], v[1] * dn[1], v[2] * dn[2]};
    const double vR[3] = {v[0] - vA[0], v[1] - vA[1], v[2] - vA[2]};
    double vC[3];
    if (d.rotLeft) { vC[0] = vR[1] * dn[2] - vR[2] * dn[1]; vC[1] = vR[2] * dn[0] - vR[0] * dn[2]; vC[2] = vR[0] * dn[1] - vR[1] * dn[0]; }
    else { vC[0] = dn[1] * vR[2] - dn[2] * vR[1]; vC[1] = dn[2] * vR[0] - dn[0] * vR[2]; vC[2] = dn[0] * vR[1] - dn[1] * vR[0]; }
    const double rLen = sqrt(vR[0] * vR[0] + vR[1] * vR[1] + vR[2] * vR[2]);
    const double cLen = sqrt(vC[0] * vC[0] + vC[1] * vC[1] + vC[2] * vC[2]);
    const double dA2 = vA[0] * vA[0] + vA[1] * vA[1] + vA[2] * vA[2];
    const double rPrime = rLen / rout, rHub = rin / rout;
    const double rStar = (rPrime - rHub) / (1.0 - rHub);
    double fR;
    if (rStar < rMin) fR = fRMin * exp(-(rStar - rMin) * (rStar - rMin) / epsR / epsR) * scale;
    else if (rStar <= rMax) fR = pow(rStar, expM) * pow(1.0 - rStar, expN) * scale;
    else fR = fRMax * exp(-(rStar - rMax) * (rStar - rMax) / epsR / epsR) * scale;
    const double fAxial = fR * exp(-dA2 / eps / eps);
    const double fCirc = fAxial * POD / 3.14159265358979323846 / (rPrime + 0.01 * eps / rout);
    for (int j = 0; j < 3; j++) out[j] += fAxial * dn[j] + (cLen > 0.0 ? fCirc * vC[j] / cLen : 0.0);
}

struct FvSourceK // fvS[j][c] = sum over the disks
{
    FvSourceSpec sp;
    const double *Cx, *Cy, *Cz;
    int nC;
    double* fvS;
    DAB_HD void operator()(int c) const
    {
        const double C[3] = {Cx[c], Cy[c], Cz[c]};
        double s[3] = {0.0, 0.0, 0.0};
        for (int k = 0; k < sp.nDisk; k++) actuatorDiskSource(sp.disk[k], C, s);
        for (int j = 0; j < 3; j++) fvS[(size_t)j * nC + c] = s[j];
    }
};

struct Params
{
    double nu, alphaU;
    double sU, sP, sNut, sPhi;           // normalizeStates
    int phiNorm;                         // "phi" is listed in normalizeStates: only then the phi rows get sPhi*|Sf| (DASolver.C:2431-2452)
    int turb, divU, divNut;              // turb: 0 laminar (dummyTurbulenceModel), 1 SpalartAllmaras
    int saFv3;                           // 1: SpalartAllmarasFv3 production term (DASpalartAllmarasFv3.C:158-175, 452-456)
    int nrU, nrP, nrNut, nrPhi;          // residual listed in normalizeResiduals
    int constrainHbyA;
    int bcKind[N_FIELDS][MAXP];
    double bcVal[N_FIELDS][MAXP][3];
    // DARhoSimpleFoam (compressible): hePsiThermo, pureMixture, perfectGas, hConst, const|sutherland transport
    // (reference DAResidual::updateThermoVars, src/adjoint/DAResidual/DAResidual.C:179-293)
    int comp;                 // 1: state ordering [U | p | T | nuTilda | phi], phi = mass flux
    int heIsE, sutherland;    // energy variable e (1) or h (0); transport model
    int divE, divEkp, nrT;    // div(phi,e|h), div(phi,Ekp|K) schemes; TRes listed in normalizeResiduals
    double Rg, Cp, muC, Pr, Prt, As, Ts, TRef, sT;
    int bcKindT[MAXP];
    double bcValT[MAXP];
    int rhoFrozen;            // primal loop only: the cell density is the stored (relaxed) field, not p/(R T)
    // simple_.transonic() (DAResidualTurboFoam.C:148-189; DARhoSimpleCFoam always): pEqn = fvm::div(phid, p) - fvm::laplacian(rho rAU, p).
    // 0 off, 1 on, 2 = preconditioner residual without the div(phid,p) term (transonicPCOption 1), 3 = on with phiRes = phi in the
    // preconditioner residual (transonicPCOption 2)
    int transonic;
    int divPhidP;             // DIV_UPWIND | DIV_LINEAR | DIV_LIMITED_LINEAR
    double phidK;             // k of "limitedLinear k"
    int turboH;               // DATurboFoam with sensibleEnthalpy: - div(Teff & U) + div(p (U - URel)) in the energy row
};

// internal working state (ghost slots appended to the cell arrays)
struct StateView
{
    const double* U;   // AoS [3*nCtot]
    const double* p;   // [nCtot]
    const double* nt;  // [nCtot] (nuTilda; unused when laminar)
    const double* phi; // [nF]
    const double* T;   // [nCtot] (compressible only)
};

// the input vector of a transpose product, field by field; on one GPU the pointers alias the caller's
// vector (reference layout), on several GPUs p/nt/phi point at working copies with ghost slots
struct PsiView
{
    const double* U;   // [3*nC]   adjoint of URes (own cell only)
    const double* p;   // [nCtot]  adjoint of pRes
    const double* nt;  // [nCtot]  adjoint of nuTildaRes
    const double* phi; // [nF]     adjoint of phiRes
    const double* T;   // [nCtot]  adjoint of TRes (compressible only)
};

// forward intermediates recorded once per state (the role of the reference's AD tape)
struct RecordView
{
    double* nut;   // [nCtot]
    double* gU;    // [9][nCtot]: gU[(j*3+i)*nCtot + c] = d_i U_j
    double* gP;    // [3][nCtot]
    double* gNt;   // [3][nCtot]
    double* rAU;   // [nCtot]
    double* HbyA;  // [3][nCtot]
    double* D0;    // [nCtot] assembled momentum diagonal (without boundary coefficients)
    double* flag;  // [nCtot] relax branch: +-1 -> |D1| branch with sign(D1); 0 -> sum-off-diagonal branch
    // compressible closures (cell values; null for DASimpleFoam)
    double *rho, *nuL, *muE, *aE, *he, *Ek; // [nCtot] density, laminar nu, rho*nuEff, alphaEff, energy variable, Ekp|K
    double* gHe;                            // [3][nCtot] grad(he)
};

// reverse intermediates (per product)
struct AdjView
{
    double* mt;    // [3][nCtot]  m~ = Mbar / V
    double* Dn;    // [nCtot]     adjoint of the relaxed diagonal
    double* Udir;  // [3][nC]     direct U adjoint from stage R1
    double* pdir;  // [nC]
    double* gPb;   // [3][nCtot]  adjoint of grad(p)
    double* gUb;   // [9][nCtot]  adjoint of grad(U)
    double* gNtb;  // [3][nCtot]  adjoint of grad(nuTilda)
    double* nutb;  // [nC]        adjoint of nut (cell value)
    double* U2;    // [3][nC]     U adjoint from stage R2
    double* nt2;   // [nC]        nuTilda adjoint from stage R2
    double* bcRefb; // [3][nC] or null: per-cell partial adjoint of the U boundary reference value of the patches in bcMask
    unsigned bcMask;
    // compressible (DARhoSimpleFoam): adjoints of the cell closures and of T
    double* gHeb;                               // [3][nCtot] adjoint of grad(he)
    double *Tdir, *cRho, *cNu, *cMuE, *cAE, *cHe, *cEk; // [nC]
};

struct FaceRef
{
    int f, n;   // face, other cell (-1 on a boundary face)
    double s;   // +1 if the cell owns the face, -1 otherwise
    bool bnd;
};

DAB_HD FaceRef faceOf(const MeshView& m, int c, int k)
{
    FaceRef r;
    const int e = m.cellFaces[(size_t)k * m.nC + c];
    if (e < 0)
    {
        r.f = -1; r.n = -1; r.s = 0.0; r.bnd = false;
        return r;
    }
    r.f = e >> 1;
    const int isN = e & 1;
    r.s = isN ? -1.0 : 1.0;
    r.bnd = r.f >= m.nIF;
    r.n = m.cellNbr[(size_t)k * m.nC + c]; // one level of indirection less than own[]/nei[] (latency-bound gathers)
    return r;
}

// the same from pre-loaded table entries
DAB_HD FaceRef faceOfE(const MeshView& m, int e, int n)
{
    FaceRef r;
    if (e < 0)
    {
        r.f = -1; r.n = -1; r.s = 0.0; r.bnd = false;
        return r;
    }
    r.f = e >> 1;
    r.s = (e & 1) ? -1.0 : 1.0;
    r.bnd = r.f >= m.nIF;
    r.n = n;
    return r;
}

// load the cell's whole row of the two ELL tables before the face loop (fixed-size meshes), so that the index loads of all
// faces are in flight together instead of one dependent round trip per face (measured on B200: product 0.855 -> 0.763 ms).
// Requesting the NEXT face's cache lines with prefetch.global.L1 on top of this was measured too and is slower (1.005 ms:
// the prefetches double the LSU transactions) -- not kept.
#define DAB_FACE_PREFETCH(NF)                                                                    \
    int e_[(NF) > 0 ? (NF) : 1], n_[(NF) > 0 ? (NF) : 1];                                        \
    if ((NF) > 0)                                                                                \
    {                                                                                            \
        _Pragma("unroll") for (int k_ = 0; k_ < (NF); k_++)                                      \
        {                                                                                        \
            e_[k_] = m.cellFaces[(size_t)k_ * m.nC + c];                                         \
            n_[k_] = m.cellNbr[(size_t)k_ * m.nC + c];                                           \
        }                                                                                        \
    }
#define DAB_FACE(NF, k) ((NF) > 0 ? faceOfE(m, e_[(NF) > 0 ? (k) : 0], n_[(NF) > 0 ? (k) : 0]) : faceOf(m, c, k))

// SA constants (reference src/adjoint/DAModel/DATurbulenceModel/DASpalartAllmaras.C:47-80)
struct SA
{
    static constexpr double sigma = 0.66666, kappa = 0.41, Cb1 = 0.1355, Cb2 = 0.622, Cw2 = 0.3, Cw3 = 2.0, Cv1 = 7.1, Cs = 0.3;
    static constexpr double Cw1 = Cb1 / (kappa * kappa) + (1.0 + Cb2) / sigma;
    static constexpr double Cv1c = Cv1 * Cv1 * Cv1;
    static constexpr double Cw3p6 = 64.0;
    static constexpr double Cv2 = 5.0; // fv3 variant
};

DAB_HD double fv1f(double chi)
{
    const double c3 = chi * chi * chi;
    return c3 * frcp(c3 + SA::Cv1c);
}
// d(nuTilda*fv1(nuTilda/nu))/d nuTilda
DAB_HD double dnut_dnt(double nt, double nu)
{
    const double chi = nt * frcp(nu), c3 = chi * chi * chi, den = c3 + SA::Cv1c, iden = frcp(den);
    const double fv1 = c3 * iden, dfv1 = 3.0 * chi * chi * SA::Cv1c * iden * iden;
    return fv1 + chi * dfv1;
}

// scaling of a phi row of a product (DASolver::normalizeGradientVec, DASolver.C:2431-2452): normalizeStates.phi * |Sf| when "phi" is
// listed in normalizeStates, otherwise the row is left alone
template <class P>
DAB_HD double phiRowScale(const P& q, double magSf) { return q.phiNorm ? q.sPhi * magSf : 1.0; }

// mixed-BC value fraction (fixedValue 1, zeroGradient 0, inletOutlet 1-pos0(phi), outletInlet pos0(phi))
DAB_HD double bcFrac(int kind, double phib)
{
    switch (kind)
    {
    case BC_FIXED_VALUE:
    case BC_NUT_LOW_RE: return 1.0;
    case BC_INLET_OUTLET: return phib >= 0.0 ? 0.0 : 1.0;
    case BC_OUTLET_INLET: return phib >= 0.0 ? 1.0 : 0.0;
    default: return 0.0;
    }
}

// scalar BC: value and snGrad; `fr` returned for the adjoint (dval/dxP = 1-fr, dsng/dxP = -fr*delta)
DAB_HD void bcScalar(int kind, double ref, double xP, double phib, double dl, double& val, double& sng, double& fr)
{
    fr = bcFrac(kind, phib);
    val = fr * ref + (1.0 - fr) * xP;
    sng = fr * (ref - xP) * dl;
}

struct BCv
{
    double val[3], sng[3], vic[3], gic[3];
};

DAB_HD void bcVector(int kind, const double* ref, const double* xP, double phib, double dl, const double* nh, BCv& b)
{
    if (kind == BC_SYMMETRY)
    {
        const double xn = nh[0] * xP[0] + nh[1] * xP[1] + nh[2] * xP[2];
        for (int k = 0; k < 3; k++)
        {
            const double an = nh[k] < 0.0 ? -nh[k] : nh[k];
            b.val[k] = xP[k] - xn * nh[k];
            b.sng[k] = -(xn * nh[k]) * dl;
            b.vic[k] = 1.0 - an;
            b.gic[k] = -(dl * an);
        }
    }
    else
    {
        const double fr = bcFrac(kind, phib);
        for (int k = 0; k < 3; k++)
        {
            b.val[k] = fr * ref[k] + (1.0 - fr) * xP[k];
            b.sng[k] = fr * (ref[k] - xP[k]) * dl;
            b.vic[k] = 1.0 - fr;
            b.gic[k] = -fr * dl;
        }
    }
}

// adjoint of bcVector w.r.t. xP given adjoints of val and sng
DAB_HD void bcVectorAdj(int kind, double phib, double dl, const double* nh, const double* valb, const double* sngb, double* xPb)
{
    if (kind == BC_SYMMETRY)
    {
        double xnb = 0.0;
        for (int k = 0; k < 3; k++) xnb -= nh[k] * (valb[k] + dl * sngb[k]);
        for (int k = 0; k < 3; k++) xPb[k] += valb[k] + nh[k] * xnb;
    }
    else
    {
        const double fr = bcFrac(kind, phib);
        for (int k = 0; k < 3; k++) xPb[k] += (1.0 - fr) * valb[k] - fr * dl * sngb[k];
    }
}

// adjoint of bcVector w.r.t. the reference value (fixedValue `value` / inletOutlet `inletValue`): val = fr*ref + ...,
// sng = fr*(ref - xP)*delta.  Used by the patchVelocity input (reference src/adjoint/DAInput/DAInputPatchVelocity.C).
DAB_HD void bcVectorRefAdj(int kind, double phib, double dl, const double* valb, const double* sngb, double* refb)
{
    if (kind == BC_SYMMETRY) return;
    const double fr = bcFrac(kind, phib);
    for (int k = 0; k < 3; k++) refb[k] += fr * (valb[k] + dl * sngb[k]);
}

// linearUpwindV (OpenFOAM linearUpwindV<vector>::correction): the explicit correction `corr` is limited along
// maxCorr = the linear-interpolation increment; out = ratio*corr with ratio in {0, 1, (corr.maxCorr)/(|corr|^2+VSMALL)}
DAB_HD void luvLimit(const double* corr, const double* maxCorr, double* out)
{
    const double s = corr[0] * corr[0] + corr[1] * corr[1] + corr[2] * corr[2];
    const double mm = corr[0] * maxCorr[0] + corr[1] * maxCorr[1] + corr[2] * maxCorr[2];
    double ratio = 1.0;
    if (s > 0.0)
    {
        if (mm < 0.0) ratio = 0.0;
        else if (s > mm) ratio = mm * frcp(s + 1e-300);
    }
    for (int j = 0; j < 3; j++) out[j] = ratio * corr[j];
}
// adjoint of luvLimit (active branch): accumulates into corrb and maxCorrb
DAB_HD void luvLimitAdj(const double* corr, const double* maxCorr, const double* outb, double* corrb, double* maxCorrb)
{
    const double s = corr[0] * corr[0] + corr[1] * corr[1] + corr[2] * corr[2];
    const double mm = corr[0] * maxCorr[0] + corr[1] * maxCorr[1] + corr[2] * maxCorr[2];
    if (s > 0.0 && mm < 0.0) return;
    if (s > 0.0 && s > mm)
    {
        const double iden = frcp(s + 1e-300), r = mm * iden;
        const double g = outb[0] * corr[0] + outb[1] * corr[1] + outb[2] * corr[2];
        const double mb = g * iden, sb = -g * mm * iden * iden;
        for (int j = 0; j < 3; j++)
        {
            corrb[j] += r * outb[j] + mb * maxCorr[j] + 2.0 * sb * corr[j];
            maxCorrb[j] += mb * corr[j];
        }
        return;
    }
    for (int j = 0; j < 3; j++) corrb[j] += outb[j];
}

// nutUSpaldingWallFunction (reference src/adjoint/DAMisc/nutUSpaldingWallFunctionDF/...DF.C:44-163): the friction
// velocity u_tau solves Spalding's law f(u_tau) = 0 by Newton iterations (relative change < 1e-14, <= 1000 iterations),
// nut_w = max(0, u_tau^2/(|dU/dn| + ROOTVSMALL) - nu).  dM = d(nut_w)/d(|U_P - U_w|) through the converged root
// (implicit-function theorem; the reference differentiates the iterations with CoDiPack, equal up to the tolerance).
DAB_HD double nutSpalding(double magUp, double dl, double nu, double& dM)
{
    const double kappa = 0.41, E = 9.8, ROOTVSMALL = 1.0e-150;
    const double y = 1.0 / dl, G = magUp * dl;
    dM = 0.0;
    double ut = sqrt(nu * G);
    if (!(ut > ROOTVSMALL)) return 0.0;
    for (int it = 0; it < 1000; it++)
    {
        const double kUu = fmin(kappa * magUp / ut, 50.0);
        const double fk = exp(kUu) - 1.0 - kUu * (1.0 + 0.5 * kUu);
        const double f = -ut * y / nu + magUp / ut + (fk - kUu * kUu * kUu / 6.0) / E;
        const double df = y / nu + magUp / (ut * ut) + kUu * fk / ut / E;
        const double un = ut + f / df;
        const double err = fabs((ut - un) / ut);
        ut = un;
        if (!(ut > ROOTVSMALL) || err < 1.0e-14) break;
    }
    if (!(ut > 0.0)) return 0.0;
    const double den = G + ROOTVSMALL;
    const double nutw = ut * ut / den - nu;
    if (!(nutw > 0.0)) return 0.0;
    const double k0 = kappa * magUp / ut;
    const bool clip = !(k0 < 50.0);
    const double k = clip ? 50.0 : k0;
    const double P = exp(k) - 1.0 - k - 0.5 * k * k;
    const double dkdm = clip ? 0.0 : kappa / ut, dkdu = clip ? 0.0 : -kappa * magUp / (ut * ut);
    const double fm = 1.0 / ut + P * dkdm / E;
    const double fu = -y / nu - magUp / (ut * ut) + P * dkdu / E;
    const double dut = -fm / fu;
    dM = 2.0 * ut * dut / den - ut * ut * dl / (den * den);
    return nutw;
}

// the same with the derivative w.r.t. the laminar viscosity as well (compressible: nu_w = mu(T_w)/rho_w is a variable)
DAB_HD double nutSpalding2(double magUp, double dl, double nu, double& dM, double& dNu)
{
    const double kappa = 0.41, E = 9.8, ROOTVSMALL = 1.0e-150;
    const double y = 1.0 / dl, G = magUp * dl;
    dM = 0.0;
    dNu = 0.0;
    double ut = sqrt(nu * G);
    if (!(ut > ROOTVSMALL)) return 0.0;
    for (int it = 0; it < 1000; it++)
    {
        const double kUu = fmin(kappa * magUp / ut, 50.0);
        const double fk = exp(kUu) - 1.0 - kUu * (1.0 + 0.5 * kUu);
        const double f = -ut * y / nu + magUp / ut + (fk - kUu * kUu * kUu / 6.0) / E;
        const double df = y / nu + magUp / (ut * ut) + kUu * fk / ut / E;
        const double un = ut + f / df;
        const double err = fabs((ut - un) / ut);
        ut = un;
        if (!(ut > ROOTVSMALL) || err < 1.0e-14) break;
    }
    if (!(ut > 0.0)) return 0.0;
    const double den = G + ROOTVSMALL;
    const double nutw = ut * ut / den - nu;
    if (!(nutw > 0.0)) return 0.0;
    const double k0 = kappa * magUp / ut;
    const bool clip = !(k0 < 50.0);
    const double k = clip ? 50.0 : k0;
    const double P = exp(k) - 1.0 - k - 0.5 * k * k;
    const double dkdm = clip ? 0.0 : kappa / ut, dkdu = clip ? 0.0 : -kappa * magUp / (ut * ut);
    const double fm = 1.0 / ut + P * dkdm / E;
    const double fu = -y / nu - magUp / (ut * ut) + P * dkdu / E;
    const double fn = ut * y / (nu * nu);
    dM = 2.0 * ut * (-fm / fu) / den - ut * ut * dl / (den * den);
    dNu = 2.0 * ut * (-fn / fu) / den - 1.0;
    return nutw;
}

// nut boundary value for the BC kinds without a wall function (the variant the common kernels are compiled with)
DAB_HD double nutBoundaryBasic(int kind, double ref, double nutP, double ntB, double nu, double& dP, double& dNb)
{
    dP = 0.0;
    dNb = 0.0;
    switch (kind)
    {
    case BC_FIXED_VALUE:
    case BC_NUT_LOW_RE: return ref;
    case BC_CALCULATED: dNb = dnut_dnt(ntB, nu); return ntB * fv1f(ntB / nu);
    case BC_NUT_SPALDING: return 0.0; // unreachable: kernels with a wall function use nutBoundary<true>
    default: dP = 1.0; return nutP; // symmetry, zeroGradient
    }
}

// nut boundary value from the nut BC kind; returns d(nut_b)/d(nut_P) in dP, d(nut_b)/d(nuTilda_b) in dNb and
// d(nut_b)/d(U_P) in dU[3] (wall functions)
template <bool WF>
DAB_HD double nutBoundary(int kind, double ref, double nutP, double ntB, double nu, const double* Uc, const double* Ub, double dl,
                          double& dP, double& dNb, double* dU)
{
    dP = 0.0;
    dNb = 0.0;
    dU[0] = dU[1] = dU[2] = 0.0;
    switch (kind)
    {
    case BC_FIXED_VALUE:
    case BC_NUT_LOW_RE: return ref;
    case BC_CALCULATED: dNb = dnut_dnt(ntB, nu); return ntB * fv1f(ntB / nu);
    case BC_NUT_SPALDING:
    if (WF)
    {
        const double d[3] = {Uc[0] - Ub[0], Uc[1] - Ub[1], Uc[2] - Ub[2]};
        const double magUp = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
        double dM;
        const double v = nutSpalding(magUp, dl, nu, dM);
        if (magUp > 0.0)
            for (int j = 0; j < 3; j++) dU[j] = dM * d[j] / magUp;
        return v;
    }
    return 0.0;
    default: dP = 1.0; return nutP; // symmetry, zeroGradient
    }
}

} // namespace dab
