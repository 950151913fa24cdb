// dab::Solver -- orchestration of the adjoint hot path on one GPU (one process per GPU).
//
// Mirrors, for this path, the reference's DASolver (reference src/adjoint/DASolver/DASolver.H:55-850):
//   construction        DASolver::DASolver + DASimpleFoam::initSolver  (DASolver.C:35-118, DASimpleFoam.C:81-121)
//   updateOFFields      DASolver::updateOFFields                       (DASolver.C:1291-1300)
//   getResiduals        DASolver::calcResiduals                        (DASolver.C:2847-2861)
//   dRdWTMatVec         DASolver::dRdWTMatVecMultFunction              (DASolver.C:1364-1409)
//   calcJacTVecProduct  DASolver::calcJacTVecProduct                   (DASolver.C:1690-1839)
//   solveLinearEqn      DASolver::solveLinearEqn / DALinearEqn         (DASolver.C:1121-1155, DALinearEqn.C:28-437)
#pragma once
#include "backend.hpp"
#include "mesh.hpp"
#include "views.hpp"
#include "fwd_kernels.hpp"
#include "rev_kernels.hpp"
#include "comp_kernels.hpp"
#include "comp_rev_kernels.hpp"
#include "krylov.hpp"
#include "primal_kernels.hpp"
#include "geom_kernels.hpp"
#include "comp_primal_kernels.hpp"
#include "partition.hpp"
#include "comm.hpp"
#include <chrono>
#include <cstdlib>
#include <cstdio>
#include <fstream>
#include <map>
#include <sys/stat.h>
#include <set>

namespace dab
{

#if !defined(DAB_HOSTSIM)
#ifndef DAB_REVB_MINBLOCKS
#define DAB_REVB_MINBLOCKS 3
#endif
#ifndef DAB_FWDB_MINBLOCKS
#define DAB_FWDB_MINBLOCKS 3
#endif
template <int NF, int FEAT> struct LaunchTraits<RevB<NF, FEAT>> { static constexpr int minBlocks = DAB_REVB_MINBLOCKS; };
// measured with the hoisted load blocks (profiles/r02_kernel_experiments.md): RevA 96 registers / 5 CTAs per SM, RevC 128 / 4
template <int NF> struct LaunchTraits<RevA<NF>> { static constexpr int minBlocks = 5; };
template <int NF> struct LaunchTraits<RevC<NF>> { static constexpr int minBlocks = 4; };
template <int NF, int FEAT> struct LaunchTraits<FwdB<NF, FEAT>> { static constexpr int minBlocks = DAB_FWDB_MINBLOCKS; };
template <int NF, int FEAT> struct LaunchTraits<UEqnAssemble<NF, FEAT>> { static constexpr int minBlocks = DAB_FWDB_MINBLOCKS; };
template <int NF> struct LaunchTraits<NutEqnAssemble<NF>> { static constexpr int minBlocks = 4; };
template <int NF> struct LaunchTraits<cFwdB<NF>> { static constexpr int minBlocks = 2; };
template <int NF> struct LaunchTraits<cUEqnAssemble<NF>> { static constexpr int minBlocks = 2; };
template <int NF> struct LaunchTraits<cEEqnAssemble<NF>> { static constexpr int minBlocks = 3; };
template <int NF> struct LaunchTraits<cNutEqnAssemble<NF>> { static constexpr int minBlocks = 3; };
template <int NF> struct LaunchTraits<cPEqnAssemble<NF>> { static constexpr int minBlocks = 4; };
template <int NF> struct LaunchTraits<cPhiUpdate<NF>> { static constexpr int minBlocks = 4; };
// resident CTAs per SM of the compressible reverse kernels, measured on the 1M-cell DATurboFoam passage (profiles/r02_kernel_experiments.md):
// cRevA 2 / 3 / 4 CTAs: 0.233 / 0.233 / 0.192 ms; cRevB 2 / 3: 0.581 / 0.551 (168 registers, 1.3 KB of spills, still faster);
// cRevE (+cRevC) 2 / 3 / 4: 0.823 / 0.639 / 0.592 -- these kernels wait on gathers: more warps beat fewer spills
#ifndef DAB_CREVA_MINBLOCKS
#define DAB_CREVA_MINBLOCKS 4
#endif
#ifndef DAB_CREVB_MINBLOCKS
#define DAB_CREVB_MINBLOCKS 3
#endif
#ifndef DAB_CREVE_MINBLOCKS
#define DAB_CREVE_MINBLOCKS 4
#endif
template <int NF> struct LaunchTraits<cRevB<NF>> { static constexpr int minBlocks = DAB_CREVB_MINBLOCKS; };
template <int NF> struct LaunchTraits<cRevA<NF>> { static constexpr int minBlocks = DAB_CREVA_MINBLOCKS; };
template <int NF> struct LaunchTraits<cRevE<NF>> { static constexpr int minBlocks = DAB_CREVE_MINBLOCKS; };
template <int NF> struct LaunchTraits<cRevC<NF>> { static constexpr int minBlocks = 4; };
template <int NF> struct LaunchTraits<cFwdE<NF>> { static constexpr int minBlocks = 4; };
template <int NF> struct LaunchTraits<cFwdC<NF>> { static constexpr int minBlocks = 4; };
#endif

// DAInputPatchVelocity (reference src/adjoint/DAInput/DAInputPatchVelocity.C): input = (|U|, angle of attack in degrees)
struct PatchVelocityDef
{
    std::string name;
    std::vector<int> patches;
    int flowAxis = 0, normalAxis = 1;
    double Umag = 0.0, aoaDeg = 0.0; // last assigned values (DAGlobalVar::patchVelocity role)
};

// DAInputPatchVar (reference src/adjoint/DAInput/DAInputPatchVar.C): the boundary reference value of one field on some patches
struct PatchVarDef
{
    std::string name, varName;
    int field = -1;   // F_U, F_P, F_NUTILDA, or -2 for T
    int nComp = 1;
    std::vector<int> patches;
};

struct FunctionDef
{
    std::string name, type;              // type: force | moment | totalPressure | massFlowRate | totalPressureRatio
    std::vector<int> patches;
    std::vector<int> inletPatches, outletPatches; // totalPressureRatio (DAFunctionTotalPressureRatio.C:33-34)
    double gamma = 1.4;                  // totalPressureRatio: mixture.thermodynamics.gamma
    std::string dirMode = "fixedDirection"; // fixedDirection | parallelToFlow | normalToFlow (DAFunctionForce.C:37-70)
    std::string patchVelocityInput;      // input whose angle of attack steers the direction
    double dir[3] = {1.0, 0.0, 0.0};     // force direction / moment axis
    double center[3] = {0.0, 0.0, 0.0};  // moment centre
    double scale = 1.0;
};

// work data of the volCoord input (solver_volcoord.hpp)
struct VolCoord
{
    bool ready = false;
    int radius = 6;         // residual rows within `radius` cells of a point's home cell may depend on the point
    double relStep = 3e-5;  // finite-difference step relative to the shortest edge at the point
    int nColours = 0, maxSlots = 1;
    std::vector<int> homeStart, listStart;
    DevBuf<int32_t> dFOff, dFLab, dSlotPoint, dHomes, dLists, dLabelA, dLabelB;
    DevBuf<double> dEps, dPts, dPts0, dR2, dOut, dF1, dF2;
};

struct Solver
{
    Backend be;
    HostMesh hm;
    Params par;
    std::string solverName, caseDirectory;
    int rank = 0, nRanks = 1;
    bool partitioned = false; // the local mesh has ghost cells: several ranks, or cyclic patches (whose images are ghosts even on one rank)
    bool ghosted() const { return partitioned; }
    // options
    int gmresRestart = 1000, gmresMaxIters = 1000, useMGSO = 0, pcFillLevel = 0, printInfo = 0;
    std::string kspType = "gmres"; // adjEqnOption.kspType (extension): gmres (the reference's KSP) | idrs (IDR(s), short recurrences)
    int idrS = 4;
    int pcSymbolicOnly = 0;
    int fpMaxIters = 1000;      // adjEqnOption fpMaxIters / fpRelTol / fpMinResTolDiff (reference pyDAFoam.py:540-542)
    double fpRelTol = 1e-6, fpMinResTolDiff = 1e2, fpOmega = 0.5;
    int coarseSparseAP = 1;   // keep the columns A*(P e_a) the probing computes and apply v - A P yc as a sparse product (0: matrix-free product per application)
    int coarseProbeReach = 6; // cell levels a pressure perturbation reaches through the transposed Jacobian (coloured probing of the coarse operator; 0 = one product per aggregate)
    int transonicPCOption = -1; // reference pyDAFoam.py:394-396 (-1 none, 1 no div(phid,p) in the PC residual, 2 phiRes = phi there)
    // adjEqnOption.pcPattern (extension): "uniform" = every state of a cell is coupled to every cell residual within pcConLevel cell levels
    // and to the phi residuals of its own faces; "stateInfo" = the reference's per-(residual, state) connectivity levels
    // (DAStateInfoSimpleFoam.C:75-99, DASpalartAllmaras.C:364-373, capped by maxResConLv4JacPCMat, pyDAFoam.py:568-582) -- DASimpleFoam only
    std::string pcPattern = "uniform";
    int pcBlockCells = 0;          // > 0: block-Jacobi ILU with the natural cell order inside blocks of that many consecutive cells (PCASM overlap 0 + natural-order PCILU), level-scheduled
    int pcExtraColourRadius = 0;   // extra colouring radius of the ILU ordering (0: the minimum that keeps same-colour rows independent)
    int globalPCIters = 0;         // Richardson sweeps wrapped around the preconditioner (reference adjEqnOption.globalPCIters)
    double richardsonOmega = 1.0;
    double gmresRelTol = 1e-6, gmresAbsTol = 1e-14, gmresTolDiff = 1e2, fdStep = 1e-6;
    std::string pcType = "ilu";
    std::string pcStorage = "fp64"; // adjEqnOption.pcStorage (extension): "fp32" keeps an fp32 copy of the ILU factors for the applications
    int coarseAggregates = 0; // > 0: two-level preconditioner with that many pressure aggregates (global)
    int pcConLevel = 2; // cell-to-cell connectivity level of dRdWTPC (maxResConLv4JacPCMat role)
    std::vector<FunctionDef> functions;
    std::vector<PatchVelocityDef> patchVelocities;
    std::vector<PatchVarDef> patchVars;
    // fvSource (actuator disks) and the fvSourcePar inputs that address its parameters
    FvSourceSpec fvSpec{};
    std::vector<std::string> diskNames;
    struct FvSourceParDef { std::string name, disk; std::vector<int> indices; };
    std::vector<FvSourceParDef> fvSourcePars;
    DevBuf<double> dFvS;
    // MRF zone (constant/MRFProperties + constant/polyMesh/cellZones; reference src/adjoint/DAMisc/MRFDF)
    struct MrfZone
    {
        bool on = false;
        std::string zone;
        double omega[3] = {0, 0, 0}, origin[3] = {0, 0, 0};
        std::vector<unsigned char> cell, type, faceIn; // [nCtot], [nBF], [nF]
    } mrf;
    DevBuf<unsigned char> dMrfCell, dMrfType, dMrfFaceIn;
    DevBuf<double> dMrfFlux;
    void updateMrfFlux()
    {
        if (mrf.on) be.launch(hm.nF, MrfFluxK{mv, dMrfFaceIn.p, dMrfFlux.p});
    }

    // device mesh
    DevBuf<int32_t> dOwn, dNei, dCellFaces, dCellNbr, dBPatch;
    DevBuf<double> dS[3], dMagSf, dW, dDelta, dK[3], dCf[3], dC[3], dV, dY;
    MeshView mv;
    // state (internal working copies with ghost slots) and external-layout mirror
    DevBuf<double> dWext, dU, dP, dNt, dPhi, dT;
    DevBuf<double> rRho, rNuL, rMuE, rAE, rHe, rEk, rGHe; // compressible closures
    DevBuf<double> aGHeb, aTdir, aCRho, aCNu, aCMuE, aCAE, aCHe, aCEk;
    StateView sv;
    // forward record and reverse work arrays
    DevBuf<double> rNut, rGU, rGP, rGNt, rRAU, rHbyA, rD0, rFlag;
    RecordView rv;
    DevBuf<double> aMt, aDn, aUdir, aPdir, aGPb, aGUb, aGNtb, aNutb, aU2, aNt2;
    AdjView av;
    DevBuf<double> dR, dX, dY2; // residual / product scratch in external layout
    bool recorded = false;
    Krylov kry;
    // domain decomposition (one rank per GPU)
    Comm comm;
    Halo halo;
    Partition part;
    DevBuf<double> psiP, psiN, psiPhi, psiT; // working copies of the input vector with ghost slots (multi-rank only)

    bool fvSourceDirty = false;
    bool hex6 = false; // every owned cell has exactly 6 faces: the kernels with fully unrolled, break-free face loops apply
    int nCellStates() const { return 4 + (par.comp ? 1 : 0) + (par.turb ? 1 : 0); }
    int nDof() const { return nCellStates() * hm.nC + hm.nF; }
    void requireIncompressible(const char* what) const
    {
        if (par.comp) throw Error(std::string(what) + ": not available for DARhoSimpleFoam yet (the forward residual is; DESIGN.md section 8)");
    }

    // bit 0: div(phi,U) is linearUpwindV; bit 1: some patch carries a wall-function nut BC
    int featureMask() const
    {
        int f = par.divU == DIV_LINEAR_UPWIND_V ? 1 : 0;
        if (par.turb)
            for (size_t p = 0; p < hm.patches.size(); p++)
                if (par.bcKind[F_NUT][p] == BC_NUT_SPALDING) f |= 2;
        if (av.bcRefb) f = 7; // patchVelocity product: the full-featured variant also carries the BC-reference adjoint
        return f;
    }

    // launch F<NF>{a...} over the cells [0, n): hexahedral meshes (6 faces per cell) get fully unrolled face loops (NF = 6),
    // anything else the run-time loop (NF = 0)
    template <template <int> class F, class... A>
    void launchNF(int n, const A&... a)
    {
        if (hex6) be.launch(n, F<6>{a...});
        else be.launch(n, F<0>{a...});
    }
    // the same with the optional-feature dispatch of the two heavy kernels (hex meshes: 4 variants; other meshes: the full-featured one)
    template <template <int, int> class F, class... A>
    void launchNFF(int n, const A&... a)
    {
        if (!hex6)
        {
            be.launch(n, F<0, 7>{a...});
            return;
        }
        switch (featureMask())
        {
        case 0: be.launch(n, F<6, 0>{a...}); break;
        case 1: be.launch(n, F<6, 1>{a...}); break;
        case 2: be.launch(n, F<6, 2>{a...}); break;
        case 3: be.launch(n, F<6, 3>{a...}); break;
        default: be.launch(n, F<6, 7>{a...}); break;
        }
    }
    // the same launches over the cell range [c0, c0 + n) (interior / cut-adjacent split for communication overlap)
    template <template <int> class F, class... A>
    void launchNFRange(int c0, int n, const A&... a)
    {
        if (hex6) be.launch(n, Shifted<F<6>>{F<6>{a...}, c0});
        else be.launch(n, Shifted<F<0>>{F<0>{a...}, c0});
    }
    template <template <int, int> class F, class... A>
    void launchNFFRange(int c0, int n, const A&... a)
    {
        if (!hex6)
        {
            be.launch(n, Shifted<F<0, 7>>{F<0, 7>{a...}, c0});
            return;
        }
        switch (featureMask())
        {
        case 0: be.launch(n, Shifted<F<6, 0>>{F<6, 0>{a...}, c0}); break;
        case 1: be.launch(n, Shifted<F<6, 1>>{F<6, 1>{a...}, c0}); break;
        case 2: be.launch(n, Shifted<F<6, 2>>{F<6, 2>{a...}, c0}); break;
        case 3: be.launch(n, Shifted<F<6, 3>>{F<6, 3>{a...}, c0}); break;
        default: be.launch(n, Shifted<F<6, 7>>{F<6, 7>{a...}, c0}); break;
        }
    }

    // ------------------------------------------------------------------------------------------
    void create(const std::string& caseDir, const std::string& argsAll, const std::string& optionsJson, int device, int rank_,
                int nRanks_, const void* ncclUid)
    {
        rank = rank_;
        nRanks = nRanks_;
        caseDirectory = caseDir;
        {
            auto t = tokenize(argsAll);
            solverName = t.empty() ? "DASimpleFoam" : t[0];
        }
        if (solverName != "DASimpleFoam" && solverName != "DARhoSimpleFoam" && solverName != "DATurboFoam" && solverName != "DARhoSimpleCFoam")
            throw Error("solver " + solverName + " is not supported (DASimpleFoam, DARhoSimpleFoam, DARhoSimpleCFoam, DATurboFoam)");
        be.init(device);
        auto tPrev = std::chrono::steady_clock::now();
        const bool setupInfo = getenv("DAB_SETUP_INFO") != nullptr;
        auto lap = [&](const char* what) {
            const auto now = std::chrono::steady_clock::now();
            if (setupInfo) fprintf(stderr, "[dab200] setup %-28s %.3f s (rank %d)\n", what, std::chrono::duration<double>(now - tPrev).count(), rank);
            tPrev = now;
        };
        hm.read(caseDir);
        lap("read polyMesh");
        bool correctWalls = false; // option wallDistCorrectWalls (OpenFOAM wallDist correctWalls): needed before the other options are applied
        if (!optionsJson.empty())
        {
            const JVal o = parseJson(optionsJson);
            if (o.kind == JVal::Obj) correctWalls = o.numOr("wallDistCorrectWalls", 0.0) != 0.0;
        }
        partitioned = nRanks > 1 || hm.hasCyclic();
        if (!partitioned)
        {
            hm.computeGeometry();
            lap("geometry");
            hm.computeWallDistance();
            if (correctWalls) hm.correctWallDistance();
            lap("wall distance");
            part.nGlobalCells = hm.nC;
        }
        else
        {
            // every rank reads the whole case, partitions it identically (RCB) and keeps its own sub-mesh; a mesh with cyclic patches
            // takes this route on one rank too (the periodic images of its cells are ghost cells, partition.hpp)
            HostMesh g;
            std::swap(g, hm);
            g.computeGeometry();
            lap("geometry (global)");
            std::vector<int> cellPart;
            rcbPartition(g, nRanks, cellPart);
            lap("RCB partition");
            {
                // wall distance of this rank's cells and their face neighbours (the ghosts) against ALL wall faces of the global mesh
                std::vector<uint8_t> mine(g.nC, 0);
                for (int c = 0; c < g.nC; c++) mine[c] = cellPart[c] == rank;
                for (int f = 0; f < g.nIF; f++)
                {
                    const int a = g.own[f], b = g.nei[f];
                    if (cellPart[a] == rank) mine[b] = 1;
                    if (cellPart[b] == rank) mine[a] = 1;
                }
                g.computeWallDistance(&mine);
                if (correctWalls) g.correctWallDistance(&mine);
            }
            lap("wall distance (own cells)");
            extractLocalMesh(g, cellPart, rank, nRanks, hm, part);
            lap("local sub-mesh");
            if (nRanks > 1) comm.initNccl(be, rank, nRanks, ncclUid);
            halo.build(be, comm, part.halo, hm.xforms);
            lap("NCCL + halo plans");
        }
        if ((int)hm.patches.size() > MAXP) throw Error("too many patches");
        readCase(caseDir);
        readMrf(caseDir);
        if (mrf.on)
            for (int b = 0; b < hm.nBF; b++)
                if (mrf.type[b] == 1 && par.bcKind[F_U][hm.bPatch[b]] != BC_FIXED_VALUE)
                    throw Error("MRF: patch " + hm.patches[hm.bPatch[b]].name
                                + " rotates with the zone and needs a fixedValue U (list it in nonRotatingPatches otherwise)");
        lap("dictionaries");
        applyOptions(optionsJson, true);
        upload();
        lap("upload");
        initialStates(caseDir);
        lap("initial states");
    }

    static int bcKindOf(const std::string& t, const std::string& where)
    {
        if (t == "fixedValue") return BC_FIXED_VALUE;
        if (t == "zeroGradient") return BC_ZERO_GRADIENT;
        if (t == "inletOutlet") return BC_INLET_OUTLET;
        if (t == "outletInlet") return BC_OUTLET_INLET;
        if (t == "symmetry" || t == "symmetryPlane") return BC_SYMMETRY;
        if (t == "calculated") return BC_CALCULATED;
        if (t == "nutLowReWallFunction") return BC_NUT_LOW_RE;
        if (t == "nutUSpaldingWallFunction" || t == "nutUSpaldingWallFunctionDF") return BC_NUT_SPALDING;
        throw Error("unsupported boundary condition type '" + t + "' in " + where);
    }

    std::map<std::string, Dict> fieldDicts;

    // one active zone of constant/MRFProperties; the face classification is MRFZoneDF::setMRFFaces (MRFZoneDF.C)
    void readMrf(const std::string& caseDir)
    {
        mrf = MrfZone();
        if (!fileExists(caseDir + "/constant/MRFProperties")) return;
        Dict d = readDict(caseDir + "/constant/MRFProperties");
        const Dict* z = nullptr;
        for (const auto& kv : d.subs)
        {
            if (kv.first == "FoamFile") continue;
            const std::string act = kv.second.wordOr("active", "true");
            if (act == "false" || act == "no" || act == "off") continue;
            if (z) throw Error("MRFProperties: more than one active zone is not supported");
            z = &kv.second;
        }
        if (!z) return;
        mrf.on = true;
        mrf.zone = z->word("cellZone");
        double ax[3] = {0, 0, 1};
        z->uniform("axis", ax);
        z->uniform("origin", mrf.origin);
        const double om = z->scalarOr("omega", 0.0), an = std::sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]);
        for (int k = 0; k < 3; k++) mrf.omega[k] = om * ax[k] / an;
        std::vector<std::string> nonRot;
        if (z->has("nonRotatingPatches"))
            for (const auto& t : z->tokens("nonRotatingPatches"))
                if (t != "(" && t != ")") nonRot.push_back(t);
        // the zone's cells (global labels)
        const std::string czPath = caseDir + "/constant/polyMesh/cellZones";
        if (!fileExists(czPath)) throw Error("cannot find MRF cellZone " + mrf.zone + " (no constant/polyMesh/cellZones)");
        const std::string txt = readFile(czPath);
        if (txt.find("format") != std::string::npos && txt.find("binary") != std::string::npos && txt.find("binary") < txt.find("}"))
            throw Error("cellZones: binary format is not supported");
        const std::vector<std::string> t = tokenize(txt);
        std::vector<unsigned char> gmask((size_t)part.nGlobalCells, 0);
        bool found = false;
        for (size_t i = 0; i + 1 < t.size() && !found; i++)
        {
            if (t[i] != mrf.zone || t[i + 1] != "{") continue;
            size_t j = i + 2;
            while (j < t.size() && t[j] != "cellLabels") j++;
            while (j < t.size() && t[j] != "(") j++;
            for (j++; j < t.size() && t[j] != ")"; j++)
            {
                const long c = atol(t[j].c_str());
                if (c < 0 || c >= (long)gmask.size()) throw Error("cellZones: cell label out of range");
                gmask[c] = 1;
            }
            found = true;
        }
        if (!found) throw Error("cannot find MRF cellZone " + mrf.zone);
        const int nT = hm.nCtot, nIF = hm.nIF;
        mrf.cell.assign(nT, 0);
        for (int c = 0; c < nT; c++) mrf.cell[c] = gmask[partitioned ? (size_t)part.cellGlobal[c] : (size_t)c];
        mrf.type.assign(hm.nBF, 0);
        mrf.faceIn.assign(hm.nF, 0);
        for (int f = 0; f < nIF; f++)
            if (mrf.cell[hm.own[f]] || mrf.cell[hm.nei[f]]) mrf.faceIn[f] = 1;
        for (int b = 0; b < hm.nBF; b++)
        {
            if (!mrf.cell[hm.own[nIF + b]]) continue;
            const std::string& pn = hm.patches[hm.bPatch[b]].name;
            const bool excluded = std::find(nonRot.begin(), nonRot.end(), pn) != nonRot.end();
            mrf.type[b] = excluded ? 2 : 1;
            if (excluded) mrf.faceIn[nIF + b] = 1;
        }
    }

    void readCase(const std::string& caseDir)
    {
        memset(&par, 0, sizeof(par));
        par.comp = solverName == "DASimpleFoam" ? 0 : 1;
        if (!par.comp)
        {
            Dict tp = readDict(caseDir + "/constant/transportProperties");
            par.nu = tp.scalar("nu");
        }
        else
        {
            // constant/thermophysicalProperties: the combination DAResidual::updateThermoVars assumes (DAResidual.C:179-293)
            Dict th = readDict(caseDir + "/constant/thermophysicalProperties");
            const Dict& tt = th.sub("thermoType");
            if (tt.wordOr("type", "hePsiThermo") != "hePsiThermo" || tt.wordOr("equationOfState", "perfectGas") != "perfectGas"
                || tt.wordOr("thermo", "hConst") != "hConst")
                throw Error("thermophysicalProperties: only hePsiThermo / perfectGas / hConst is supported");
            const std::string en = tt.wordOr("energy", "sensibleInternalEnergy"), trn = tt.wordOr("transport", "const");
            if (en != "sensibleInternalEnergy" && en != "sensibleEnthalpy") throw Error("thermophysicalProperties: unsupported energy " + en);
            if (trn != "const" && trn != "sutherland") throw Error("thermophysicalProperties: unsupported transport " + trn);
            par.heIsE = en == "sensibleInternalEnergy" ? 1 : 0;
            par.turboH = (solverName == "DATurboFoam" && !par.heIsE) ? 1 : 0;
            par.sutherland = trn == "sutherland" ? 1 : 0;
            const Dict& mx = th.sub("mixture");
            par.Rg = 8314.4700665 / mx.sub("specie").scalar("molWeight");
            par.Cp = mx.sub("thermodynamics").scalar("Cp");
            gammaTPR = mx.sub("thermodynamics").scalarOr("gamma", par.Cp / (par.Cp - par.Rg));
            const Dict& tr = mx.sub("transport");
            par.muC = tr.scalarOr("mu", 1.8e-5);
            par.Pr = tr.scalarOr("Pr", 0.7);
            par.As = tr.scalarOr("As", 1.4792e-6);
            par.Ts = tr.scalarOr("Ts", 116.0);
            par.Prt = th.scalarOr("Prt", 1.0);
            par.TRef = 298.15;
            par.sT = 1.0;
            par.nrT = 1;
            par.nu = par.muC; // unused by the compressible kernels
        }
        std::string ras = "dummy";
        if (fileExists(caseDir + "/constant/turbulenceProperties"))
        {
            Dict tu = readDict(caseDir + "/constant/turbulenceProperties");
            if (tu.hasSub("RAS")) ras = tu.sub("RAS").wordOr("RASModel", "dummy");
        }
        if (ras == "SpalartAllmaras") par.turb = 1;
        else if (ras == "SpalartAllmarasFv3") { par.turb = 1; par.saFv3 = 1; }
        else if (ras == "dummy" || ras == "dummyTurbulenceModel" || ras == "laminar") par.turb = 0;
        else throw Error("RASModel " + ras + " is not supported (SpalartAllmaras, SpalartAllmarasFv3, dummy)");
        Dict fs = readDict(caseDir + "/system/fvSchemes");
        auto scheme = [&](const std::string& key) {
            std::string v = fs.sub("divSchemes").joined(key);
            // the steady solvers of the reference run `bounded Gauss ...` convection (boundedConvectionScheme: - fvm::Sp(div(phi)));
            // the kernels have that form built in
            if (v.find("bounded") == std::string::npos)
                throw Error("divSchemes " + key + " '" + v + "': only 'bounded Gauss <scheme>' is supported");
            if (v.find("linearUpwindV") != std::string::npos)
            {
                if (key != "div(phi,U)") throw Error("linearUpwindV applies to vector fields only (" + key + ")");
                return (int)DIV_LINEAR_UPWIND_V;
            }
            if (v.find("linearUpwind") != std::string::npos) return (int)DIV_LINEAR_UPWIND;
            if (v.find("upwind") != std::string::npos) return (int)DIV_UPWIND;
            if (v.find("linear") != std::string::npos) return (int)DIV_LINEAR;
            throw Error("unsupported div scheme '" + v + "'");
        };
        par.divU = scheme("div(phi,U)");
        par.divNut = par.turb ? scheme("div(phi,nuTilda)") : DIV_UPWIND;
        if (par.comp)
        {
            par.divE = scheme(par.heIsE ? "div(phi,e)" : "div(phi,h)");
            par.divEkp = scheme(par.heIsE ? "div(phi,Ekp)" : "div(phi,K)");
            if (par.divEkp != DIV_UPWIND && par.divEkp != DIV_LINEAR) throw Error("div(phi,Ekp|K): upwind or linear");
            // temperature boundary conditions
            const std::string path = caseDir + "/0/T";
            Dict d = readDict(path);
            fieldDicts["T"] = d;
            const Dict& bf = d.sub("boundaryField");
            for (size_t p = 0; p < hm.patches.size(); p++)
            {
                const Dict& pd = bf.sub(hm.patches[p].name);
                const int kind = bcKindOf(pd.word("type"), path);
                par.bcKindT[p] = kind;
                double v[3] = {0, 0, 0};
                const char* key = kind == BC_INLET_OUTLET ? "inletValue" : (kind == BC_OUTLET_INLET ? "outletValue" : "value");
                if (pd.has(key)) pd.uniform(key, v);
                par.bcValT[p] = v[0];
            }
        }
        Dict fso = readDict(caseDir + "/system/fvSolution");
        par.alphaU = 1.0;
        if (fso.hasSub("relaxationFactors") && fso.sub("relaxationFactors").hasSub("equations"))
            par.alphaU = fso.sub("relaxationFactors").sub("equations").scalarOr("U", 1.0);
        if (fso.hasSub("SIMPLE"))
        {
            const std::string c = fso.sub("SIMPLE").wordOr("consistent", "false");
            primal.consistent = (c == "true" || c == "yes" || c == "on");
        }
        // transonic pressure equation: SIMPLE { transonic yes; } (simpleControl::transonic()); DARhoSimpleCFoam has no other form
        // (DAResidualRhoSimpleCFoam.C:160 "we don't support transonic = false")
        par.transonic = 0;
        par.divPhidP = DIV_UPWIND;
        par.phidK = 1.0;
        if (par.comp)
        {
            std::string tr = fso.hasSub("SIMPLE") ? fso.sub("SIMPLE").wordOr("transonic", "no") : "no";
            if (solverName == "DARhoSimpleCFoam" || tr == "yes" || tr == "true" || tr == "on")
            {
                par.transonic = 1;
                const std::string v = fs.sub("divSchemes").joined("div(phid,p)");
                const size_t ll = v.find("limitedLinear");
                if (ll != std::string::npos)
                {
                    par.divPhidP = DIV_LIMITED_LINEAR;
                    par.phidK = atof(v.c_str() + ll + 13);
                    if (!(par.phidK > 0.0 && par.phidK <= 1.0)) throw Error("div(phid,p) '" + v + "': limitedLinear needs 0 < k <= 1");
                }
                else if (v.find("linearUpwind") != std::string::npos)
                    throw Error("div(phid,p) '" + v + "': upwind, linear or limitedLinear k");
                else if (v.find("upwind") != std::string::npos) par.divPhidP = DIV_UPWIND;
                else if (v.find("linear") != std::string::npos) par.divPhidP = DIV_LINEAR;
                else throw Error("div(phid,p) '" + v + "': upwind, linear or limitedLinear k");
            }
        }
        if (solverName == "DATurboFoam") primal.consistent = true; // its pressure corrector always uses AtU = AU - H1 (pEqnTurbo.H:13)
        // primal solver controls (system/fvSolution, system/controlDict)
        if (fso.hasSub("relaxationFactors"))
        {
            const Dict& rf = fso.sub("relaxationFactors");
            if (rf.hasSub("fields")) primal.alphaP = rf.sub("fields").scalarOr("p", primal.alphaP);
            if (rf.hasSub("fields")) primal.alphaRho = rf.sub("fields").scalarOr("rho", primal.alphaRho);
            if (rf.hasSub("equations")) primal.alphaN = rf.sub("equations").scalarOr("nuTilda", primal.alphaN);
            if (rf.hasSub("equations"))
                primal.alphaE = rf.sub("equations").scalarOr("e", rf.sub("equations").scalarOr("h", primal.alphaE));
        }
        if (fso.hasSub("SIMPLE")) primal.nNonOrth = (int)fso.sub("SIMPLE").scalarOr("nNonOrthogonalCorrectors", 0.0);
        if (fso.hasSub("solvers"))
        {
            const Dict& sd = fso.sub("solvers");
            auto ctl = [&](const char* name, SegControl& c) {
                if (!sd.hasSub(name)) return;
                c.tol = sd.sub(name).scalarOr("tolerance", c.tol);
                c.relTol = sd.sub(name).scalarOr("relTol", c.relTol);
                c.maxIter = (int)sd.sub(name).scalarOr("maxIter", (double)c.maxIter);
            };
            ctl("U", primal.cU);
            ctl("p", primal.cP);
            ctl("nuTilda", primal.cN);
            ctl("e", primal.cE);
            ctl("h", primal.cE);
        }
        if (fileExists(caseDir + "/system/controlDict"))
        {
            Dict cd = readDict(caseDir + "/system/controlDict");
            const double endTime = cd.scalarOr("endTime", 1000.0), deltaT = cd.scalarOr("deltaT", 1.0), startTime = cd.scalarOr("startTime", 0.0);
            primal.maxIters = (int)((endTime - startTime) / deltaT + 0.5);
        }
        // boundary conditions
        const char* fn[N_FIELDS] = {"U", "p", "nuTilda", "nut"};
        for (int fi = 0; fi < N_FIELDS; fi++)
        {
            if (fi >= F_NUTILDA && !par.turb) continue;
            const std::string path = caseDir + "/0/" + fn[fi];
            Dict d = readDict(path);
            fieldDicts[fn[fi]] = d;
            const Dict& bf = d.sub("boundaryField");
            for (size_t p = 0; p < hm.patches.size(); p++)
            {
                const Dict& pd = bf.sub(hm.patches[p].name);
                const std::string ty = pd.word("type");
                const int kind = bcKindOf(ty, path);
                par.bcKind[fi][p] = kind;
                double v[3] = {0, 0, 0};
                const char* key = kind == BC_INLET_OUTLET ? "inletValue" : (kind == BC_OUTLET_INLET ? "outletValue" : "value");
                if (pd.has(key)) pd.uniform(key, v);
                for (int k = 0; k < 3; k++) par.bcVal[fi][p][k] = v[k];
            }
        }
        // defaults of the reference's DAOPTION (dafoam/pyDAFoam.py:526-563)
        par.sU = par.sP = par.sNut = par.sPhi = 1.0;
        par.phiNorm = 0; // normalizeStates is empty by default: no state is scaled
        par.nrU = par.nrP = par.nrNut = par.nrPhi = 1;
        par.constrainHbyA = 1;
    }

    void applyOptions(const std::string& json, bool first)
    {
        if (json.empty()) return;
        JVal o = parseJson(json);
        if (o.kind != JVal::Obj) throw Error("options must be a JSON object");
        if (const JVal* ns = o.get("normalizeStates"))
        {
            par.sU = ns->numOr("U", par.sU);
            par.sP = ns->numOr("p", par.sP);
            par.sNut = ns->numOr("nuTilda", par.sNut);
            par.sPhi = ns->numOr("phi", par.sPhi);
            par.phiNorm = ns->get("phi") ? 1 : 0;
            par.sT = ns->numOr("T", par.sT);
        }
        if (const JVal* nr = o.get("normalizeResiduals"))
        {
            par.nrU = par.nrP = par.nrNut = par.nrPhi = par.nrT = 0;
            for (const auto& v : nr->arr)
            {
                if (v.str == "URes") par.nrU = 1;
                if (v.str == "pRes") par.nrP = 1;
                if (v.str == "nuTildaRes") par.nrNut = 1;
                if (v.str == "phiRes") par.nrPhi = 1;
                if (v.str == "TRes") par.nrT = 1;
            }
        }
        par.constrainHbyA = (int)o.numOr("useConstrainHbyA", par.constrainHbyA);
        {
            const int tpo = (int)o.numOr("transonicPCOption", transonicPCOption);
            if (tpo != transonicPCOption) { transonicPCOption = tpo; kry.pcValid = false; }
        }
        if (const JVal* a = o.get("adjEqnOption"))
        {
            gmresRestart = (int)a->numOr("gmresRestart", gmresRestart);
            gmresMaxIters = (int)a->numOr("gmresMaxIters", gmresMaxIters);
            gmresRelTol = a->numOr("gmresRelTol", gmresRelTol);
            gmresAbsTol = a->numOr("gmresAbsTol", gmresAbsTol);
            gmresTolDiff = a->numOr("gmresTolDiff", gmresTolDiff);
            useMGSO = (int)a->numOr("useMGSO", useMGSO);
            pcFillLevel = (int)a->numOr("pcFillLevel", pcFillLevel);
            printInfo = (int)a->numOr("printInfo", printInfo);
            pcType = a->strOr("pcType", pcType);
            {
                const std::string ps = a->strOr("pcStorage", pcStorage);
                if (ps != "fp64" && ps != "fp32") throw Error("adjEqnOption.pcStorage " + ps + ": fp64 or fp32");
                if (ps != pcStorage) { pcStorage = ps; kry.pcValid = false; }
            }
            pcSymbolicOnly = (int)a->numOr("pcSymbolicOnly", pcSymbolicOnly);
            fpMaxIters = (int)a->numOr("fpMaxIters", fpMaxIters);
            fpRelTol = a->numOr("fpRelTol", fpRelTol);
            fpMinResTolDiff = a->numOr("fpMinResTolDiff", fpMinResTolDiff);
            fpOmega = a->numOr("fpOmega", fpOmega);
            {
                const int sa = (int)a->numOr("coarseSparseAP", coarseSparseAP);
                if (sa != coarseSparseAP) { coarseSparseAP = sa; kry.pcValid = false; }
            }
            {
                const int pr = (int)a->numOr("coarseProbeReach", coarseProbeReach);
                if (pr != coarseProbeReach) { coarseProbeReach = pr; kry.pcValid = false; }
            }
            kspType = a->strOr("kspType", kspType);
            if (kspType != "gmres" && kspType != "idrs") throw Error("adjEqnOption.kspType " + kspType + ": gmres or idrs");
            idrS = (int)a->numOr("idrS", idrS);
            if (idrS < 1 || idrS > 16) throw Error("adjEqnOption.idrS: 1..16");
            globalPCIters = (int)a->numOr("globalPCIters", globalPCIters);
            {
                const std::string pp = a->strOr("pcPattern", pcPattern);
                if (pp != "uniform" && pp != "stateInfo") throw Error("adjEqnOption.pcPattern " + pp + ": uniform or stateInfo");
                if (pp != pcPattern) { pcPattern = pp; kry.symbolic = false; kry.pcValid = false; }
                const int bc = (int)a->numOr("pcBlockCells", pcBlockCells);
                if (bc != pcBlockCells) { pcBlockCells = bc; kry.symbolic = false; kry.pcValid = false; }
            }
            {
                const int cr = (int)a->numOr("pcColourRadius", pcExtraColourRadius);
                if (cr != pcExtraColourRadius) { pcExtraColourRadius = cr; kry.symbolic = false; kry.pcValid = false; }
            }
            richardsonOmega = a->numOr("richardsonOmega", richardsonOmega);
            const int ca = (int)a->numOr("coarseAggregates", coarseAggregates);
            if (ca != coarseAggregates) { coarseAggregates = ca; kry.pcValid = false; }
            const int lv = (int)a->numOr("pcConLevel", pcConLevel);
            if (lv != pcConLevel) { pcConLevel = lv; kry.symbolic = false; kry.pcValid = false; }
        }
        if (const JVal* s = o.get("adjPartDerivFDStep"))
        {
            fdStep = s->numOr("State", fdStep);
            volc.relStep = s->numOr("Coord", volc.relStep); // relative to the shortest edge at the point
        }
        primal.minResTol = o.numOr("primalMinResTol", primal.minResTol);
        primal.minResTolDiff = o.numOr("primalMinResTolDiff", primal.minResTolDiff);
        primal.minIters = (int)o.numOr("primalMinIters", primal.minIters);
        primal.maxIters = (int)o.numOr("primalMaxIters", primal.maxIters); // extension: overrides controlDict endTime/deltaT
        primal.printInterval = (int)o.numOr("printInterval", primal.printInterval);
        if (const JVal* ps = o.get("primalSolver")) // extension: controls of the device pressure solver
        {
            primal.nAgg = (int)ps->numOr("coarseAggregates", primal.nAgg);
            primal.coarseRefresh = std::max(1, (int)ps->numOr("coarseRefresh", primal.coarseRefresh));
            primal.alphaRho = ps->numOr("rhoRelax", primal.alphaRho);
            primal.alphaE = ps->numOr("heRelax", primal.alphaE);
            primal.alphaP = ps->numOr("pRelax", primal.alphaP);
        }
        if (const JVal* vb = o.get("primalVarBounds"))
        {
            primal.ntMin = vb->numOr("nuTildaMin", primal.ntMin);
            primal.ntMax = vb->numOr("nuTildaMax", primal.ntMax);
            primal.pMin = vb->numOr("pMin", primal.pMin);
            primal.pMax = vb->numOr("pMax", primal.pMax);
            primal.TMin = vb->numOr("TMin", primal.TMin);
            primal.TMax = vb->numOr("TMax", primal.TMax);
            primal.UMax = vb->numOr("UMax", primal.UMax);
        }
        adjPCLag = (int)o.numOr("adjPCLag", (double)adjPCLag);
        if (const JVal* wj = o.get("writeJacobians"))
        {
            keepPCMatrix = false;
            for (const auto& v : wj->arr)
                if (v.str == "dRdWTPC" || v.str == "all") keepPCMatrix = true;
        }
        if (const JVal* pb = o.get("primalBC"))
        {
            // DAField::setPrimalBoundaryConditions (reference DAField.C:698-1260): boundary values, nut wall treatment, MRF speed
            // and the laminar viscosity from the options, applied before the primal solution
            for (const auto& kv : pb->obj)
            {
                const std::string& key = kv.first;
                if (key == "useWallFunction")
                {
                    const bool wf = kv.second.kind == JVal::Bool ? kv.second.b : kv.second.num != 0.0;
                    for (size_t p = 0; p < hm.patches.size(); p++)
                        if (hm.patchGeom[p] == PG_WALL && par.turb) par.bcKind[F_NUT][p] = wf ? BC_NUT_SPALDING : BC_NUT_LOW_RE;
                    continue;
                }
                if (key == "MRF")
                {
                    if (!mrf.on) throw Error("primalBC.MRF: the case has no MRF zone");
                    const double mg = std::sqrt(mrf.omega[0] * mrf.omega[0] + mrf.omega[1] * mrf.omega[1] + mrf.omega[2] * mrf.omega[2]);
                    if (mg == 0.0) throw Error("primalBC.MRF: omega 0 in MRFProperties leaves the sense of rotation undefined");
                    for (int k = 0; k < 3; k++)
                    {
                        mrf.omega[k] *= kv.second.num / mg;
                        mv.mrfOmega[k] = mrf.omega[k];
                    }
                    if (dMrfFlux.p) updateMrfFlux();
                    continue;
                }
                if (key == "transport:nu")
                {
                    if (par.comp) throw Error("primalBC transport:nu: incompressible solvers only");
                    par.nu = kv.second.num;
                    continue;
                }
                if (key == "thermo:mu")
                {
                    if (!par.comp) throw Error("primalBC thermo:mu: compressible solvers only");
                    par.muC = kv.second.num;
                    continue;
                }
                if (kv.second.kind != JVal::Obj) throw Error("primalBC." + key + " is not supported");
                const std::string var = kv.second.strOr("variable", "");
                const JVal* val = kv.second.get("value");
                const JVal* pl = kv.second.get("patches");
                if (!val || !pl) throw Error("primalBC." + key + ": patches, variable and value are required");
                if (val->arr.size() != 1 && val->arr.size() != 3)
                    throw Error("value should be a list of either 1 (scalar) or 3 (vector) elements");
                int field = -1;
                if (var == "U") field = F_U;
                else if (var == "p") field = F_P;
                else if (var == "nuTilda") field = F_NUTILDA;
                else if (var == "nut") field = F_NUT;
                const bool isT = var == "T";
                if (field < 0 && !isT) continue; // "<variable> not found, skip it."
                if ((field == F_U) != (val->arr.size() == 3)) throw Error("primalBC." + key + ": value size does not fit " + var);
                if ((isT && !par.comp) || (field == F_NUTILDA && !par.turb)) continue;
                for (const auto& pn : pl->arr)
                {
                    int p = -1;
                    for (size_t q = 0; q < hm.patches.size(); q++)
                        if (hm.patches[q].name == pn.str) p = (int)q;
                    if (p < 0) throw Error("primalBC." + key + ": unknown patch " + pn.str);
                    const int kind = isT ? par.bcKindT[p] : par.bcKind[field][p];
                    if (kind != BC_FIXED_VALUE && kind != BC_INLET_OUTLET && kind != BC_OUTLET_INLET)
                        throw Error("only support fixedValues, inletOutlet, outletInlet");
                    if (isT) par.bcValT[p] = val->arr[0].num;
                    else
                        for (size_t k = 0; k < val->arr.size(); k++) par.bcVal[field][p][k] = val->arr[k].num;
                }
            }
            recorded = false;
            kry.pcValid = false;
        }
        if (const JVal* fd = o.get("function"))
        {
            functions.clear();
            for (const auto& kv : fd->obj)
            {
                FunctionDef f;
                f.name = kv.first;
                f.type = kv.second.strOr("type", "force");
                if (f.type != "force" && f.type != "moment" && f.type != "totalPressure" && f.type != "massFlowRate"
                    && f.type != "totalPressureRatio")
                    throw Error("function type " + f.type + " is not supported (force, moment, totalPressure, massFlowRate, totalPressureRatio)");
                auto patchList = [&](const char* key, std::vector<int>& out) {
                    if (const JVal* pl = kv.second.get(key))
                        for (const auto& pn : pl->arr)
                        {
                            int found = -1;
                            for (size_t p = 0; p < hm.patches.size(); p++)
                                if (hm.patches[p].name == pn.str) found = (int)p;
                            if (found < 0) throw Error("function " + f.name + ": unknown patch " + pn.str);
                            out.push_back(found);
                        }
                };
                patchList("patches", f.patches);
                if (f.type == "totalPressureRatio")
                {
                    if (!par.comp) throw Error("function " + f.name + ": totalPressureRatio needs a compressible solver");
                    patchList("inletPatches", f.inletPatches);
                    patchList("outletPatches", f.outletPatches);
                    for (int p : f.patches)
                        if (std::find(f.inletPatches.begin(), f.inletPatches.end(), p) == f.inletPatches.end()
                            && std::find(f.outletPatches.begin(), f.outletPatches.end(), p) == f.outletPatches.end())
                            throw Error("inlet/outletPatches names are not in patches");
                    if (f.inletPatches.empty() || f.outletPatches.empty()) throw Error("function " + f.name + ": inletPatches / outletPatches are required");
                    f.gamma = gammaTPR;
                }
                if (f.type == "moment")
                {
                    if (const JVal* d = kv.second.get("axis"))
                        for (size_t k = 0; k < 3 && k < d->arr.size(); k++) f.dir[k] = d->arr[k].num;
                    if (const JVal* d = kv.second.get("center"))
                        for (size_t k = 0; k < 3 && k < d->arr.size(); k++) f.center[k] = d->arr[k].num;
                }
                else if (f.type == "force")
                {
                    f.dirMode = kv.second.strOr("directionMode", "fixedDirection");
                    if (f.dirMode == "fixedDirection")
                    {
                        if (const JVal* d = kv.second.get("direction"))
                            for (size_t k = 0; k < 3 && k < d->arr.size(); k++) f.dir[k] = d->arr[k].num;
                    }
                    else if (f.dirMode == "parallelToFlow" || f.dirMode == "normalToFlow")
                    {
                        f.patchVelocityInput = kv.second.strOr("patchVelocityInputName", "");
                        if (f.patchVelocityInput.empty()) throw Error("function " + f.name + ": patchVelocityInputName is required");
                    }
                    else
                        throw Error("directionMode for " + f.name + " not valid! Options: fixedDirection, parallelToFlow, normalToFlow.");
                }
                const double mg = std::sqrt(f.dir[0] * f.dir[0] + f.dir[1] * f.dir[1] + f.dir[2] * f.dir[2]);
                if (std::fabs(mg - 1.0) > 1e-8) throw Error("the magnitude of the direction parameter in " + f.name + " is not 1.0!");
                f.scale = kv.second.numOr("scale", 1.0);
                functions.push_back(f);
            }
        }
        if (const JVal* fsd = o.get("fvSource"))
        {
            // DAFvSourceActuatorDisk::initFvSourcePars (reference DAFvSourceActuatorDisk.C:427-485)
            fvSpec.nDisk = 0;
            diskNames.clear();
            for (const auto& kv : fsd->obj)
            {
                if (kv.second.strOr("type", "") != "actuatorDisk" || kv.second.strOr("source", "") != "cylinderAnnulusSmooth")
                    throw Error("fvSource." + kv.first + ": only type actuatorDisk with source cylinderAnnulusSmooth is supported");
                if (kv.second.numOr("adjustThrust", 0.0) != 0.0) throw Error("fvSource." + kv.first + ": adjustThrust is not supported");
                if (fvSpec.nDisk >= MAXDISK) throw Error("too many actuator disks");
                ActuatorDisk& d = fvSpec.disk[fvSpec.nDisk++];
                diskNames.push_back(kv.first);
                const JVal* c = kv.second.get("center");
                const JVal* dr = kv.second.get("direction");
                if (!c || !dr || c->arr.size() != 3 || dr->arr.size() != 3) throw Error("fvSource." + kv.first + ": center and direction (3 numbers) are required");
                for (int k = 0; k < 3; k++) { d.par[k] = c->arr[k].num; d.par[3 + k] = dr->arr[k].num; }
                d.par[6] = kv.second.numOr("innerRadius", 0.0);
                d.par[7] = kv.second.numOr("outerRadius", 1.0);
                d.par[8] = kv.second.numOr("scale", 1.0);
                d.par[9] = kv.second.numOr("POD", 0.0);
                d.par[10] = kv.second.numOr("expM", 1.0);
                d.par[11] = kv.second.numOr("expN", 0.5);
                d.par[12] = kv.second.numOr("targetThrust", 1.0);
                d.eps = kv.second.numOr("eps", 0.1);
                const std::string rd = kv.second.strOr("rotDir", "right");
                if (rd != "left" && rd != "right") throw Error("rotDir not valid");
                d.rotLeft = rd == "left" ? 1 : 0;
            }
            fvSourceDirty = true;
        }
        if (const JVal* ii = o.get("inputInfo"))
        {
            fvSourcePars.clear();
            for (const auto& kv : ii->obj)
            {
                if (kv.second.strOr("type", "") != "fvSourcePar") continue;
                FvSourceParDef d;
                d.name = kv.first;
                d.disk = kv.second.strOr("fvSourceName", "");
                if (const JVal* il = kv.second.get("indices"))
                    for (const auto& iv : il->arr)
                    {
                        const int idx = (int)iv.num;
                        if (idx < 0 || idx > 12) throw Error("inputInfo." + kv.first + ": indices must be in 0..12");
                        d.indices.push_back(idx);
                    }
                fvSourcePars.push_back(d);
            }
            patchVars.clear();
            for (const auto& kv : ii->obj)
            {
                if (kv.second.strOr("type", "") != "patchVar") continue;
                PatchVarDef d;
                d.name = kv.first;
                d.varName = kv.second.strOr("varName", "");
                const std::string vt = kv.second.strOr("varType", "scalar");
                if (vt != "scalar" && vt != "vector") throw Error("inputInfo." + kv.first + ": varType not valid");
                d.nComp = vt == "vector" ? 3 : 1;
                if (d.varName == "U") d.field = F_U;
                else if (d.varName == "p") d.field = F_P;
                else if (d.varName == "nuTilda") d.field = F_NUTILDA;
                else if (d.varName == "T" && par.comp) d.field = -2;
                else throw Error("inputInfo." + kv.first + ": varName " + d.varName + " is not a boundary field of this solver");
                if ((d.field == F_U) != (d.nComp == 3)) throw Error("inputInfo." + kv.first + ": varType does not match " + d.varName);
                if (const JVal* pl = kv.second.get("patches"))
                    for (const auto& pn : pl->arr)
                    {
                        int found = -1;
                        for (size_t p = 0; p < hm.patches.size(); p++)
                            if (hm.patches[p].name == pn.str) found = (int)p;
                        if (found < 0) throw Error("inputInfo." + kv.first + ": unknown patch " + pn.str);
                        const int kind = d.field == -2 ? par.bcKindT[found] : par.bcKind[d.field][found];
                        if (kind != BC_FIXED_VALUE && kind != BC_INLET_OUTLET && kind != BC_OUTLET_INLET)
                            throw Error("inputInfo." + kv.first + ": patch type not valid! only support fixedValue or inletOutlet");
                        d.patches.push_back(found);
                    }
                patchVars.push_back(d);
            }
            patchVelocities.clear();
            for (const auto& kv : ii->obj)
            {
                if (kv.second.strOr("type", "") != "patchVelocity") continue;
                PatchVelocityDef d;
                d.name = kv.first;
                auto axis = [&](const std::string& a) {
                    if (a == "x") return 0;
                    if (a == "y") return 1;
                    if (a == "z") return 2;
                    throw Error("inputInfo." + kv.first + ": axis must be x, y or z");
                };
                d.flowAxis = axis(kv.second.strOr("flowAxis", "x"));
                d.normalAxis = axis(kv.second.strOr("normalAxis", "y"));
                if (const JVal* pl = kv.second.get("patches"))
                    for (const auto& pn : pl->arr)
                    {
                        int found = -1;
                        for (size_t p = 0; p < hm.patches.size(); p++)
                            if (hm.patches[p].name == pn.str) found = (int)p;
                        if (found < 0) throw Error("inputInfo." + kv.first + ": unknown patch " + pn.str);
                        d.patches.push_back(found);
                    }
                if (!d.patches.empty())
                {
                    const double uf = par.bcVal[F_U][d.patches[0]][d.flowAxis], un = par.bcVal[F_U][d.patches[0]][d.normalAxis];
                    d.Umag = std::sqrt(uf * uf + un * un);
                    d.aoaDeg = std::atan2(un, uf) * 180.0 / 3.14159265358979323846;
                }
                patchVelocities.push_back(d);
            }
        }
        (void)first;
        recorded = false;
    }

    void upload()
    {
        dOwn.upload(be, hm.own);
        dNei.upload(be, hm.nei);
        dCellFaces.upload(be, hm.cellFaces);
        hex6 = hm.maxCF == 6;
        for (size_t i = 0; i < hm.cellFaces.size() && hex6; i++)
            if (hm.cellFaces[i] < 0) hex6 = false;
        hm.buildCellNbr();
        dCellNbr.upload(be, hm.cellNbr);
        dBPatch.upload(be, hm.bPatch);
        for (int k = 0; k < 3; k++)
        {
            dS[k].upload(be, hm.Sf[k]);
            dK[k].upload(be, hm.corr[k]);
            dCf[k].upload(be, hm.Cf[k]);
            dC[k].upload(be, hm.C[k]);
        }
        dMagSf.upload(be, hm.magSf);
        dW.upload(be, hm.w);
        dDelta.upload(be, hm.delta);
        dV.upload(be, hm.V);
        dY.upload(be, hm.yWall);
        mv.nC = hm.nC; mv.nCtot = hm.nCtot; mv.nF = hm.nF; mv.nIF = hm.nIF; mv.nBF = hm.nBF; mv.maxCF = hm.maxCF;
        mv.own = dOwn.p; mv.nei = dNei.p; mv.cellFaces = dCellFaces.p; mv.cellNbr = dCellNbr.p; mv.bPatch = dBPatch.p;
        mv.Sx = dS[0].p; mv.Sy = dS[1].p; mv.Sz = dS[2].p; mv.magSf = dMagSf.p; mv.w = dW.p; mv.delta = dDelta.p;
        mv.kx = dK[0].p; mv.ky = dK[1].p; mv.kz = dK[2].p; mv.Cfx = dCf[0].p; mv.Cfy = dCf[1].p; mv.Cfz = dCf[2].p;
        mv.Cx = dC[0].p; mv.Cy = dC[1].p; mv.Cz = dC[2].p; mv.V = dV.p; mv.yWall = dY.p;
        mv.fvS = nullptr;
        mv.mrfCell = nullptr; mv.mrfType = nullptr; mv.mrfFlux = nullptr;
        if (mrf.on)
        {
            dMrfCell.upload(be, mrf.cell);
            dMrfType.upload(be, mrf.type);
            dMrfFaceIn.upload(be, mrf.faceIn);
            dMrfFlux.alloc(be, hm.nF);
            for (int k = 0; k < 3; k++)
            {
                mv.mrfOmega[k] = mrf.omega[k];
                mv.mrfOrigin[k] = mrf.origin[k];
            }
            mv.mrfCell = dMrfCell.p; mv.mrfType = dMrfType.p; mv.mrfFlux = dMrfFlux.p;
            updateMrfFlux();
        }
        fvSourceDirty = fvSpec.nDisk > 0;
        const size_t nT = hm.nCtot, nC = hm.nC, nF = hm.nF, nd = nDof();
        dWext.alloc(be, nd);
        dU.alloc(be, 3 * nT); dP.alloc(be, nT); dNt.alloc(be, nT); dPhi.alloc(be, nF);
        sv.U = dU.p; sv.p = dP.p; sv.nt = dNt.p; sv.phi = dPhi.p; sv.T = nullptr;
        rv.rho = rv.nuL = rv.muE = rv.aE = rv.he = rv.Ek = rv.gHe = nullptr;
        if (par.comp)
        {
            dT.alloc(be, nT);
            sv.T = dT.p;
            rRho.alloc(be, nT); rNuL.alloc(be, nT); rMuE.alloc(be, nT); rAE.alloc(be, nT); rHe.alloc(be, nT); rEk.alloc(be, nT);
            rGHe.alloc(be, 3 * nT);
            rv.rho = rRho.p; rv.nuL = rNuL.p; rv.muE = rMuE.p; rv.aE = rAE.p; rv.he = rHe.p; rv.Ek = rEk.p; rv.gHe = rGHe.p;
        }
        rNut.alloc(be, nT); rGU.alloc(be, 9 * nT); rGP.alloc(be, 3 * nT); rGNt.alloc(be, 3 * nT);
        rRAU.alloc(be, nT); rHbyA.alloc(be, 3 * nT); rD0.alloc(be, nT); rFlag.alloc(be, nT);
        rv.nut = rNut.p; rv.gU = rGU.p; rv.gP = rGP.p; rv.gNt = rGNt.p; rv.rAU = rRAU.p; rv.HbyA = rHbyA.p; rv.D0 = rD0.p; rv.flag = rFlag.p;
        aMt.alloc(be, 3 * nT); aDn.alloc(be, nT); aUdir.alloc(be, 3 * nC); aPdir.alloc(be, nC);
        aGPb.alloc(be, 3 * nT); aGUb.alloc(be, 9 * nT); aGNtb.alloc(be, 3 * nT); aNutb.alloc(be, nC);
        aU2.alloc(be, 3 * nC); aNt2.alloc(be, nC);
        av.mt = aMt.p; av.Dn = aDn.p; av.Udir = aUdir.p; av.pdir = aPdir.p; av.gPb = aGPb.p; av.gUb = aGUb.p;
        av.gNtb = aGNtb.p; av.nutb = aNutb.p; av.U2 = aU2.p; av.nt2 = aNt2.p;
        av.bcRefb = nullptr; av.bcMask = 0;
        av.gHeb = av.Tdir = av.cRho = av.cNu = av.cMuE = av.cAE = av.cHe = av.cEk = nullptr;
        if (par.comp)
        {
            aGHeb.alloc(be, 3 * nT); aTdir.alloc(be, nC); aCRho.alloc(be, nC); aCNu.alloc(be, nC); aCMuE.alloc(be, nC);
            aCAE.alloc(be, nC); aCHe.alloc(be, nC); aCEk.alloc(be, nC);
            av.gHeb = aGHeb.p; av.Tdir = aTdir.p; av.cRho = aCRho.p; av.cNu = aCNu.p; av.cMuE = aCMuE.p; av.cAE = aCAE.p;
            av.cHe = aCHe.p; av.cEk = aCEk.p;
        }
        dR.alloc(be, nd); dX.alloc(be, nd); dY2.alloc(be, nd);
    }

    // DASolver::calcPCMatWithFvMatrix(PCMat, turbOnly = 1) (reference DASolver.C:2888-2988 + DASpalartAllmaras::getFvMatrixFields,
    // DASpalartAllmaras.C:490-529): the block-diagonal entries dR_nuTilda/d nuTilda taken straight from the relaxed nuTilda fvMatrix
    // assembled with the `div(pc)` (upwind) convection scheme -- D() on the diagonal, lower()/upper() on the internal faces --
    // scaled by normalizeStates.nuTilda / (V when nuTildaRes is listed in normalizeResiduals), written TRANSPOSED like the
    // reference does (MatSetValues(PCMat, col, row)).  Returned as COO triplets in the local state numbering.  The non-turbulence
    // part (turbOnly = 0) aborts in the reference for the SIMPLE family (DAResidual::calcPCMatWithFvMatrix, DAResidual.C:295-300).
    void calcPCMatWithFvMatrix(int turbOnly, std::vector<int32_t>& rows, std::vector<int32_t>& cols, std::vector<double>& vals)
    {
        if (!turbOnly)
            throw Error("calcPCMatWithFvMatrix: only turbOnly = 1 is available for " + solverName
                        + " (the reference's DAResidual::calcPCMatWithFvMatrix aborts for the SIMPLE solver family)");
        rows.clear(); cols.clear(); vals.clear();
        if (!par.turb) return;
        if (par.comp) throw Error("calcPCMatWithFvMatrix: the compressible nuTilda matrix export is not built (DASimpleFoam only)");
        ensureRecorded();
        const int nC = hm.nC, nIF = hm.nIF, mcf = hm.maxCF;
        DevBuf<double> off, diag, b;
        off.alloc(be, (size_t)mcf * nC);
        diag.alloc(be, nC);
        b.alloc(be, nC);
        EqnView e{nC, mcf, 1, off.p, diag.p, b.p, mv.cellNbr};
        Params pq = par;
        pq.divNut = DIV_UPWIND; // "div(pc)"
        launchNF<NutEqnAssemble>(nC, mv, pq, sv, rv, e, primal.alphaN);
        std::vector<double> hOff((size_t)mcf * nC), hD(nC);
        be.d2h(hOff.data(), off.p, hOff.size() * sizeof(double));
        be.d2h(hD.data(), diag.p, hD.size() * sizeof(double));
        const int base = (par.comp ? 5 : 4) * nC; // local adjoint state index of nuTilda_c (state ordering)
        auto resScale = [&](int c) { return par.nrNut ? hm.V[c] : 1.0; };
        for (int c = 0; c < nC; c++)
        {
            rows.push_back(base + c);
            cols.push_back(base + c);
            vals.push_back(hD[c] * par.sNut / resScale(c));
        }
        for (int c = 0; c < nC; c++)
            for (int k = 0; k < mcf; k++)
            {
                const int en = hm.cellFaces[(size_t)k * nC + c];
                if (en < 0) break;
                const int f = en >> 1;
                if (f >= nIF) continue;
                const int n = hm.cellNbr[(size_t)k * nC + c];
                if (n < 0 || n >= nC) continue; // cut face: the other cell belongs to another rank
                // A[c][n] (upper when c owns the face, lower otherwise), stored at the transposed position (row n, column c)
                rows.push_back(base + n);
                cols.push_back(base + c);
                vals.push_back(hOff[(size_t)k * nC + c] * par.sNut / resScale(c));
            }
    }

    // initial states from the 0/ files (DASimpleFoam::initSolver createFieldsSimple.H role); phi = linear-interpolated U . Sf
    // timeName != "0": DASolver::readStateVars (DASolver.C readStateVars role) - the internal fields (and phi, when written) of
    // <case>/<timeName>/ replace the states; the boundary conditions stay those of 0/
    void initialStates(const std::string&, const std::string& timeName = "0")
    {
        const int nC = hm.nC, nF = hm.nF, nIF = hm.nIF;
        std::vector<double> W(nDof(), 0.0);
        std::map<std::string, Dict> timeDicts;
        auto internal = [&](const std::string& name, int nc, std::vector<double>& out) {
            if (timeName != "0")
            {
                const std::string path = caseDirectory + "/" + timeName + "/" + name;
                if (!fileExists(path)) throw Error("readStateVars: " + path + " does not exist");
                timeDicts[name] = readDict(path);
            }
            const Dict& d = timeName != "0" ? timeDicts.at(name) : fieldDicts.at(name);
            const auto& t = d.tokens("internalField");
            const int nT = hm.nCtot;
            out.assign((size_t)nc * nT, 0.0);
            if (t.at(0) == "uniform")
            {
                double v[3] = {0, 0, 0};
                d.uniform("internalField", v);
                for (int c = 0; c < nT; c++)
                    for (int k = 0; k < nc; k++) out[(size_t)nc * c + k] = v[k];
            }
            else
            {
                // nonuniform List<type> N ( ... )
                std::vector<double> vals;
                size_t i = 0;
                while (i < t.size() && t[i] != "(") i++;
                for (i++; i < t.size(); i++)
                {
                    if (t[i] == "(" || t[i] == ")") continue;
                    vals.push_back(atof(t[i].c_str()));
                }
                if (vals.size() < (size_t)nc * part.nGlobalCells) throw Error("internalField of " + name + " has the wrong size");
                for (int c = 0; c < nT; c++)
                {
                    const size_t gc = partitioned ? (size_t)part.cellGlobal[c] : (size_t)c;
                    for (int k = 0; k < nc; k++) out[(size_t)nc * c + k] = vals[(size_t)nc * gc + k];
                }
            }
        };
        std::vector<double> U, p, nt, Tt;
        internal("U", 3, U);
        internal("p", 1, p);
        for (int i = 0; i < 3 * nC; i++) W[i] = U[i];
        for (int c = 0; c < nC; c++) W[3 * (size_t)nC + c] = p[c];
        size_t off = 4 * (size_t)nC;
        if (par.comp)
        {
            internal("T", 1, Tt);
            for (int c = 0; c < nC; c++) W[off + c] = Tt[c];
            off += nC;
        }
        if (par.turb)
        {
            internal("nuTilda", 1, nt);
            for (int c = 0; c < nC; c++) W[off + c] = nt[c];
            off += nC;
        }
        for (int f = 0; f < nF; f++)
        {
            double uf[3];
            const int o = hm.own[f];
            if (f < nIF)
                for (int k = 0; k < 3; k++) uf[k] = hm.w[f] * U[3 * (size_t)o + k] + (1.0 - hm.w[f]) * U[3 * (size_t)hm.nei[f] + k];
            else
            {
                const int pa = hm.bPatch[f - nIF];
                const int kind = par.bcKind[F_U][pa];
                for (int k = 0; k < 3; k++) uf[k] = (kind == BC_FIXED_VALUE) ? par.bcVal[F_U][pa][k] : U[3 * (size_t)o + k];
                if (kind == BC_SYMMETRY) uf[0] = uf[1] = uf[2] = 0.0;
            }
            W[off + f] = uf[0] * hm.Sf[0][f] + uf[1] * hm.Sf[1][f] + uf[2] * hm.Sf[2][f];
            if (f >= nIF && par.bcKind[F_U][hm.bPatch[f - nIF]] == BC_SYMMETRY) W[off + f] = 0.0;
            if (par.comp)
            {
                // mass flux: rho_f from the cell values (createFieldsRhoSimple.H role)
                const double ro = p[o] / (par.Rg * Tt[o]);
                const double rf = f < nIF ? hm.w[f] * ro + (1.0 - hm.w[f]) * p[hm.nei[f]] / (par.Rg * Tt[hm.nei[f]]) : ro;
                W[off + f] *= rf;
            }
        }
        // a flux field written by a previous run (writeFields / OpenFOAM's own phi) takes precedence over the interpolated one
        if (!partitioned && fileExists(caseDirectory + "/" + timeName + "/phi"))
        {
            Dict d = readDict(caseDirectory + "/" + timeName + "/phi");
            auto listOf = [&](const std::vector<std::string>& t, size_t n, std::vector<double>& out) {
                out.clear();
                if (!t.empty() && t[0] == "uniform")
                {
                    out.assign(n, atof(t.at(1).c_str()));
                    return;
                }
                size_t i = 0;
                while (i < t.size() && t[i] != "(") i++;
                for (i++; i < t.size() && t[i] != ")"; i++) out.push_back(atof(t[i].c_str()));
                if (out.size() != n) throw Error(timeName + "/phi: a list has " + std::to_string(out.size()) + " entries, expected " + std::to_string(n));
            };
            std::vector<double> v;
            listOf(d.tokens("internalField"), (size_t)nIF, v);
            for (int f = 0; f < nIF; f++) W[off + f] = v[f];
            const Dict& bf = d.sub("boundaryField");
            for (const PatchDef& p : hm.patches)
            {
                const Dict& pd = bf.sub(p.name);
                if (!pd.has("value")) continue; // e.g. symmetry: stays zero
                listOf(pd.tokens("value"), (size_t)p.size, v);
                for (int i = 0; i < p.size; i++) W[off + p.start + i] = v[i];
            }
        }
        updateOFFields(W.data());
    }

    // ------------------------------------------------------------------------------------------
    // host mirror of the states last assigned through updateOFFields: calcJacTVecProduct(stateVar, ...) re-assigns the states on every
    // call (DAInputStateVar::run); when they are the resident ones the record and the preconditioner stay valid (ADVICE round 1: computing
    // dFdW after calcdRdWT used to force a second assembly inside the next solveLinearEqn)
    std::vector<double> hWMirror;
    bool hWMirrorValid = false;
    bool statesAreResident(const double* W) const
    {
        return hWMirrorValid && hWMirror.size() == (size_t)nDof() && std::memcmp(hWMirror.data(), W, hWMirror.size() * sizeof(double)) == 0;
    }
    void updateOFFields(const double* W)
    {
        const size_t nC = hm.nC;
        hWMirror.assign(W, W + nDof());
        hWMirrorValid = true;
        be.h2d(dWext.p, W, (size_t)nDof() * sizeof(double));
        be.d2d(dU.p, dWext.p, 3 * nC * sizeof(double));
        be.d2d(dP.p, dWext.p + 3 * nC, nC * sizeof(double));
        size_t off = 4 * nC;
        if (par.comp)
        {
            be.d2d(dT.p, dWext.p + off, nC * sizeof(double));
            off += nC;
        }
        if (par.turb)
        {
            be.d2d(dNt.p, dWext.p + off, nC * sizeof(double));
            off += nC;
        }
        be.d2d(dPhi.p, dWext.p + off, (size_t)hm.nF * sizeof(double));
        exchangeStates();
        recorded = false;
        kry.pcValid = false;
    }

    // ghost cells <- owners (U, p, nuTilda) and foreign cut faces <- owners (phi)
    void exchangeStates()
    {
        if (!ghosted()) return;
        const int nT = hm.nCtot;
        std::vector<HaloItem> it{{dU.p, 3, 3, 1}, {dP.p, 1, 1, nT}};
        if (par.turb) it.push_back({dNt.p, 1, 1, nT});
        if (par.comp) it.push_back({dT.p, 1, 1, nT});
        halo.exchangeCells(it);
        halo.exchangeFaces({{dPhi.p, 1, 1, hm.nF}});
    }

    void getOFFields(double* W) { be.d2h(W, dWext.p, (size_t)nDof() * sizeof(double)); }

    // fvSource field from the disk parameters and the current cell centres (DAFvSourceActuatorDisk::calcFvSource)
    void updateFvSource()
    {
        if (fvSpec.nDisk == 0)
        {
            mv.fvS = nullptr;
            fvSourceDirty = false;
            return;
        }
        if (dFvS.n < (size_t)3 * hm.nC) dFvS.alloc(be, (size_t)3 * hm.nC);
        be.launch(hm.nC, FvSourceK{fvSpec, mv.Cx, mv.Cy, mv.Cz, hm.nC, dFvS.p});
        mv.fvS = dFvS.p;
        fvSourceDirty = false;
        recorded = false;
        kry.pcValid = false;
    }

    int diskIndex(const std::string& name) const
    {
        for (size_t i = 0; i < diskNames.size(); i++)
            if (diskNames[i] == name) return (int)i;
        throw Error("fvSource " + name + " is not defined");
    }
    const FvSourceParDef& findFvSourcePar(const std::string& name) const
    {
        for (const auto& d : fvSourcePars)
            if (d.name == name) return d;
        throw Error("input " + name + " (fvSourcePar) is not defined in inputInfo");
    }
    void setFvSourcePar(const std::string& name, const double* in)
    {
        const FvSourceParDef& d = findFvSourcePar(name);
        ActuatorDisk& k = fvSpec.disk[diskIndex(d.disk)];
        for (size_t i = 0; i < d.indices.size(); i++) k.par[d.indices[i]] = in[i];
        updateFvSource();
    }
    // product[i] = [dR/d(par_i)]^T psi (or seed * dF/d(par_i)) by central differences on the device kernels
    void fvSourceParProduct(const std::string& name, const double* in, const double* psi, const std::string* fname, double seed, double* product)
    {
        const FvSourceParDef& d = findFvSourcePar(name);
        const size_t n = nDof();
        std::vector<double> Rp, Rm, x(in, in + d.indices.size());
        if (!fname) { Rp.resize(n); Rm.resize(n); }
        for (size_t k = 0; k < d.indices.size(); k++)
        {
            const double h = std::max(1e-6, 1e-5 * std::fabs(in[k]));
            double vp = 0.0, vm = 0.0;
            for (int sgn = 0; sgn < 2; sgn++)
            {
                std::vector<double> xx(x);
                xx[k] += sgn == 0 ? h : -h;
                setFvSourcePar(name, xx.data());
                if (fname) (sgn == 0 ? vp : vm) = calcFunction(*fname);
                else
                {
                    forward(0, dR.p);
                    be.d2h(sgn == 0 ? Rp.data() : Rm.data(), dR.p, n * sizeof(double));
                }
            }
            if (fname) product[k] = seed * (vp - vm) / (2.0 * h);
            else
            {
                double sdot = 0.0;
                for (size_t i = 0; i < n; i++) sdot += psi[i] * (Rp[i] - Rm[i]);
                product[k] = sdot / (2.0 * h);
            }
        }
        setFvSourcePar(name, in);
    }

    // forward passes; record(isPC=0) leaves the intermediates the reverse sweep reuses
    void forward(int isPC, double* Rdev, bool exchange = true)
    {
        const int nT = hm.nCtot;
        if (fvSourceDirty) updateFvSource();
        if (par.comp)
        {
            // DARhoSimpleFoam: closures + gradients, momentum/SA rows, energy row, pressure/flux rows (comp_kernels.hpp)
            launchNF<cFwdA>(hm.nCtot, mv, par, sv, rv); // closures of the ghost cells come from their exchanged states
            if (exchange && ghosted())
            {
                std::vector<HaloItem> it{{rv.gU, 9, 1, nT}, {rv.gP, 3, 1, nT}, {rv.gHe, 3, 1, nT}};
                if (par.turb) it.push_back({rv.gNt, 3, 1, nT});
                halo.exchangeCells(it);
            }
            launchNF<cFwdB>(hm.nC, mv, par, sv, rv, isPC, Rdev);
            launchNF<cFwdE>(hm.nC, mv, par, sv, rv, isPC, Rdev);
            if (exchange && ghosted()) halo.exchangeCells({{rv.rAU, 1, 1, nT}, {rv.HbyA, 3, 1, nT}, {rv.flag, 1, 1, nT}});
            if (isPC && par.transonic)
            {
                Params pq = par; // div(pc) scheme and transonicPCOption for the preconditioner residual
                pq.divPhidP = DIV_UPWIND;
                pq.transonic = transonicPCOption == 1 ? 2 : (transonicPCOption == 2 ? 3 : 1);
                launchNF<cFwdC>(hm.nC, mv, pq, sv, rv, Rdev);
            }
            else
                launchNF<cFwdC>(hm.nC, mv, par, sv, rv, Rdev);
            return;
        }
        launchNF<FwdA>(hm.nCtot, mv, par, sv, rv);
        if (exchange && ghosted())
        {
            std::vector<HaloItem> it{{rv.gU, 9, 1, nT}, {rv.gP, 3, 1, nT}};
            if (par.turb) it.push_back({rv.gNt, 3, 1, nT});
            halo.exchangeCells(it);
        }
        launchNFF<FwdB>(hm.nC, mv, par, sv, rv, isPC, Rdev);
        if (exchange && ghosted()) halo.exchangeCells({{rv.rAU, 1, 1, nT}, {rv.HbyA, 3, 1, nT}, {rv.flag, 1, 1, nT}});
        launchNF<FwdC>(hm.nC, mv, par, sv, rv, Rdev);
    }

    void ensureRecorded()
    {
        if (recorded) return;
        forward(0, dR.p);
        recorded = true;
    }

    void getResiduals(int isPC, double* R)
    {
        forward(isPC, dR.p);
        recorded = (isPC == 0);
        be.d2h(R, dR.p, (size_t)nDof() * sizeof(double));
    }

    PsiView psiView(const double* x)
    {
        const size_t nC = hm.nC;
        PsiView v;
        v.U = x;
        v.T = nullptr;
        if (!ghosted())
        {
            v.p = x + 3 * nC;
            v.T = par.comp ? x + 4 * nC : nullptr;
            v.nt = x + (par.comp ? 5 : 4) * nC;
            v.phi = x + (size_t)nCellStates() * nC;
            return v;
        }
        const int nT = hm.nCtot;
        if (psiP.n < (size_t)nT)
        {
            psiP.alloc(be, nT);
            psiN.alloc(be, nT);
            psiPhi.alloc(be, hm.nF);
        }
        be.d2d(psiP.p, x + 3 * nC, nC * sizeof(double));
        std::vector<HaloItem> it{{psiP.p, 1, 1, nT}};
        if (par.comp)
        {
            if (psiT.n < (size_t)nT) psiT.alloc(be, nT);
            be.d2d(psiT.p, x + 4 * nC, nC * sizeof(double));
            it.push_back({psiT.p, 1, 1, nT});
            v.T = psiT.p;
        }
        if (par.turb)
        {
            be.d2d(psiN.p, x + (par.comp ? 5 : 4) * nC, nC * sizeof(double));
            it.push_back({psiN.p, 1, 1, nT});
        }
        be.d2d(psiPhi.p, x + (size_t)nCellStates() * nC, (size_t)hm.nF * sizeof(double));
        halo.exchangeCells(it);
        halo.exchangeFaces({{psiPhi.p, 1, 1, hm.nF}});
        v.p = psiP.p;
        v.nt = psiN.p;
        v.phi = psiPhi.p;
        return v;
    }

    // y = diag(n) (dR/dW)^T x on device vectors (external layout)
    void matVecDev(const double* x, double* y)
    {
        ensureRecorded();
        if (par.comp)
        {
            // DARhoSimpleFoam reverse sweep (comp_rev_kernels.hpp), one GPU
            const PsiView pv = psiView(x);
            const int nTc = hm.nCtot;
            launchNF<cRevA>(hm.nC, mv, par, sv, rv, av, pv);
            if (ghosted()) halo.exchangeCells({{av.mt, 3, 1, nTc}, {av.Dn, 1, 1, nTc}, {av.gPb, 3, 1, nTc}});
            launchNF<cRevB>(hm.nC, mv, par, sv, rv, av, pv, y);
            launchNF<cRevE>(hm.nC, mv, par, sv, rv, av, pv, y);
            if (ghosted())
            {
                std::vector<HaloItem> it{{av.gUb, 9, 1, nTc}, {av.gHeb, 3, 1, nTc}};
                if (par.turb) it.push_back({av.gNtb, 3, 1, nTc});
                halo.exchangeCells(it);
            }
            launchNF<cRevC>(hm.nC, mv, par, sv, rv, av, y);
            return;
        }
        const int nT = hm.nCtot;
        if (!ghosted())
        {
            const PsiView pv = psiView(x);
            launchNF<RevA>(hm.nC, mv, par, sv, rv, av, pv);
            launchNFF<RevB>(hm.nC, mv, par, sv, rv, av, pv, y);
            launchNF<RevC>(hm.nC, mv, par, sv, rv, av, y, 0);
            return;
        }
        // several ranks: every ghost exchange runs on the communication stream while the interior cells (no neighbour on
        // another rank) of the next stage are processed; the cut-adjacent cells follow once the ghosts have arrived
        const int nI = hm.nInterior < 0 ? hm.nC : hm.nInterior, nB = hm.nC - nI;
        const PsiView pv = psiViewStart(x);
        launchNFRange<RevA>(0, nI, mv, par, sv, rv, av, pv);
        halo.finish();
        launchNFRange<RevA>(nI, nB, mv, par, sv, rv, av, pv);
        halo.start(halo.cells, {{av.mt, 3, 1, nT}, {av.Dn, 1, 1, nT}, {av.gPb, 3, 1, nT}});
        launchNFFRange<RevB>(0, nI, mv, par, sv, rv, av, pv, y);
        halo.finish();
        launchNFFRange<RevB>(nI, nB, mv, par, sv, rv, av, pv, y);
        {
            std::vector<HaloItem> it{{av.gUb, 9, 1, nT}};
            if (par.turb) it.push_back({av.gNtb, 3, 1, nT});
            halo.start(halo.cells, it);
        }
        launchNFRange<RevC>(0, nI, mv, par, sv, rv, av, y, 0);
        halo.finish();
        launchNFRange<RevC>(nI, nB, mv, par, sv, rv, av, y, 0);
    }

    // ghost values of the input vector, exchange started but not awaited (halo.finish() before the first reader)
    PsiView psiViewStart(const double* x)
    {
        const size_t nC = hm.nC;
        const int nT = hm.nCtot;
        if (psiP.n < (size_t)nT)
        {
            psiP.alloc(be, nT);
            psiN.alloc(be, nT);
            psiPhi.alloc(be, hm.nF);
        }
        PsiView v;
        v.U = x;
        be.d2d(psiP.p, x + 3 * nC, nC * sizeof(double));
        std::vector<HaloItem> it{{psiP.p, 1, 1, nT}};
        if (par.turb)
        {
            be.d2d(psiN.p, x + 4 * nC, nC * sizeof(double));
            it.push_back({psiN.p, 1, 1, nT});
        }
        be.d2d(psiPhi.p, x + (par.turb ? 5 : 4) * nC, (size_t)hm.nF * sizeof(double));
        halo.start(halo.cells, it);
        halo.start(halo.faces, {{psiPhi.p, 1, 1, hm.nF}});
        v.p = psiP.p;
        v.nt = psiN.p;
        v.phi = psiPhi.p;
        return v;
    }

    // one reverse kernel alone on the bench vectors (dab_bench_device selectors 2-4).  On several ranks the kernel runs over all owned
    // cells on the ghost values the last full product left behind: no copy, no exchange inside the timed launches
    void benchKernel(int which)
    {
        PsiView pv;
        if (ghosted() && psiP.n >= (size_t)hm.nCtot)
        {
            pv.U = dX.p; pv.p = psiP.p; pv.nt = psiN.p; pv.phi = psiPhi.p; pv.T = psiT.n ? psiT.p : nullptr;
        }
        else
            pv = psiView(dX.p);
        if (par.comp)
        {
            // DARhoSimpleFoam: 0 cRevA, 1 cRevB, 2 cRevE + cRevC
            if (which == 0) launchNF<cRevA>(hm.nC, mv, par, sv, rv, av, pv);
            else if (which == 1) launchNF<cRevB>(hm.nC, mv, par, sv, rv, av, pv, dY2.p);
            else
            {
                launchNF<cRevE>(hm.nC, mv, par, sv, rv, av, pv, dY2.p);
                launchNF<cRevC>(hm.nC, mv, par, sv, rv, av, dY2.p);
            }
            return;
        }
        if (which == 0) launchNF<RevA>(hm.nC, mv, par, sv, rv, av, pv);
        else if (which == 1) launchNFF<RevB>(hm.nC, mv, par, sv, rv, av, pv, dY2.p);
        else launchNF<RevC>(hm.nC, mv, par, sv, rv, av, dY2.p, 0);
    }

    void matVec(const double* x, double* y)
    {
        be.h2d(dX.p, x, (size_t)nDof() * sizeof(double));
        matVecDev(dX.p, dY2.p);
        be.d2h(y, dY2.p, (size_t)nDof() * sizeof(double));
    }

    // ---- patchVelocity input (DAInputPatchVelocity::run + its reverse) --------------------------------
    const PatchVelocityDef& findPatchVelocity(const std::string& name) const
    {
        for (const auto& d : patchVelocities)
            if (d.name == name) return d;
        throw Error("input " + name + " (patchVelocity) is not defined in inputInfo");
    }

    // assign (|U|, aoa[deg]) to the U boundary reference values of the patches
    void setPatchVelocity(const std::string& name, const double* in)
    {
        PatchVelocityDef& d = const_cast<PatchVelocityDef&>(findPatchVelocity(name));
        d.Umag = in[0];
        d.aoaDeg = in[1];
        const double a = in[1] * 3.14159265358979323846 / 180.0;
        for (int p : d.patches)
        {
            par.bcVal[F_U][p][d.flowAxis] = in[0] * std::cos(a);
            par.bcVal[F_U][p][d.normalAxis] = in[0] * std::sin(a);
        }
        recorded = false;
        kry.pcValid = false;
    }

    DevBuf<double> aBcRefb;

    // ---- patchVar input (DAInputPatchVar): assignment and products by central differences on the device kernels
    const PatchVarDef& findPatchVar(const std::string& name) const
    {
        for (const auto& d : patchVars)
            if (d.name == name) return d;
        throw Error("input " + name + " (patchVar) is not defined in inputInfo");
    }
    void setPatchVar(const std::string& name, const double* in)
    {
        const PatchVarDef& d = findPatchVar(name);
        for (int p : d.patches)
        {
            if (d.field == -2) par.bcValT[p] = in[0];
            else
                for (int k = 0; k < d.nComp; k++) par.bcVal[d.field][p][k] = in[k];
        }
        recorded = false;
        kry.pcValid = false;
    }
    double patchVarStep(const PatchVarDef& d, double x) const
    {
        const double sc = d.field == F_U ? par.sU : (d.field == F_P ? par.sP : (d.field == F_NUTILDA ? par.sNut : par.sT));
        // compromise between the round-off of psi.(R+ - R-) (R ~ 1e6 for compressible cases) and the kinks of the limited schemes:
        // accurate to ~1e-4; the exact alternative is the BC-reference adjoint of the reverse kernels (patchVelocity has it)
        return std::max(1e-6 * std::fabs(sc), 1e-4 * std::fabs(x));
    }
    // product[nComp] = [dR/d(value)]^T psi, or seed * dF/d(value) when fname is given
    void patchVarProduct(const std::string& name, const double* in, const double* psi, const std::string* fname, double seed, double* product)
    {
        const PatchVarDef& d = findPatchVar(name);
        const size_t n = nDof();
        std::vector<double> Rp, Rm, x(in, in + d.nComp);
        if (!fname) { Rp.resize(n); Rm.resize(n); }
        for (int k = 0; k < d.nComp; k++)
        {
            const double h = patchVarStep(d, in[k]);
            double vp = 0.0, vm = 0.0;
            for (int sgn = 0; sgn < 2; sgn++)
            {
                std::vector<double> xx(x);
                xx[k] += sgn == 0 ? h : -h;
                setPatchVar(name, xx.data());
                if (fname) (sgn == 0 ? vp : vm) = calcFunction(*fname);
                else
                {
                    forward(0, dR.p);
                    be.d2h(sgn == 0 ? Rp.data() : Rm.data(), dR.p, n * sizeof(double));
                }
            }
            if (fname) product[k] = seed * (vp - vm) / (2.0 * h);
            else
            {
                double sdot = 0.0;
                for (size_t i = 0; i < n; i++) sdot += psi[i] * (Rp[i] - Rm[i]);
                if (ghosted())
                {
                    be.h2d(dY2.p, &sdot, sizeof(double));
                    comm.allreduceSum(be, dY2.p, 1);
                    be.d2h(&sdot, dY2.p, sizeof(double));
                }
                product[k] = sdot / (2.0 * h);
            }
        }
        setPatchVar(name, in);
    }

    // product[2] = [dR/d(|U|, aoa)]^T psi
    void patchVelocityProduct(const std::string& name, const double* in, const double* psi, double* product)
    {
        const PatchVelocityDef& d = findPatchVelocity(name);
        setPatchVelocity(name, in);
        if (par.comp)
        {
            // DARhoSimpleFoam: two scalar inputs -> central differences of psi . R on the device kernels (4 residual evaluations,
            // O(eps^2)); the BC-reference adjoint of the incompressible reverse kernels is the exact alternative
            const size_t n = nDof();
            std::vector<double> Rp(n), Rm(n);
            const double h[2] = {1e-6 * std::max(1.0, std::fabs(in[0])), 1e-6};
            for (int k = 0; k < 2; k++)
            {
                double xp[2] = {in[0], in[1]}, xm[2] = {in[0], in[1]};
                xp[k] += h[k];
                xm[k] -= h[k];
                setPatchVelocity(name, xp);
                forward(0, dR.p);
                be.d2h(Rp.data(), dR.p, n * sizeof(double));
                setPatchVelocity(name, xm);
                forward(0, dR.p);
                be.d2h(Rm.data(), dR.p, n * sizeof(double));
                double sdot = 0.0;
                for (size_t i = 0; i < n; i++) sdot += psi[i] * (Rp[i] - Rm[i]);
                product[k] = sdot / (2.0 * h[k]);
            }
            setPatchVelocity(name, in);
            return;
        }
        const size_t nC = hm.nC;
        if (aBcRefb.n < 3 * nC) aBcRefb.alloc(be, 3 * nC);
        unsigned mask = 0;
        for (int p : d.patches) mask |= 1u << p;
        be.h2d(dX.p, psi, (size_t)nDof() * sizeof(double));
        av.bcRefb = aBcRefb.p;
        av.bcMask = mask;
        matVecDev(dX.p, dY2.p);
        av.bcRefb = nullptr;
        av.bcMask = 0;
        std::vector<double> part(3 * nC);
        be.d2h(part.data(), aBcRefb.p, 3 * nC * sizeof(double));
        double refb[3] = {0, 0, 0};
        for (int k = 0; k < 3; k++)
            for (size_t c = 0; c < nC; c++) refb[k] += part[k * nC + c];
        if (ghosted())
        {
            be.h2d(aBcRefb.p, refb, 3 * sizeof(double));
            comm.allreduceSum(be, aBcRefb.p, 3);
            be.d2h(refb, aBcRefb.p, 3 * sizeof(double));
        }
        const double a = in[1] * 3.14159265358979323846 / 180.0;
        product[0] = refb[d.flowAxis] * std::cos(a) + refb[d.normalAxis] * std::sin(a);
        product[1] = (-refb[d.flowAxis] * in[0] * std::sin(a) + refb[d.normalAxis] * in[0] * std::cos(a)) * 3.14159265358979323846 / 180.0;
    }

    // ---- functions (DAFunctionForce) ------------------------------------------------------------
    const FunctionDef& findFunction(const std::string& name) const
    {
        for (const auto& f : functions)
            if (f.name == name) return f;
        throw Error("function " + name + " is not defined in the options");
    }

    // dAlpha = true: the direction is replaced by its derivative w.r.t. the angle of attack [rad]
    ForceSpec forceSpec(const FunctionDef& f, bool dAlpha = false) const
    {
        ForceSpec fs;
        fs.mask = 0;
        for (int p : f.patches) fs.mask |= (1u << p);
        for (int k = 0; k < 3; k++) { fs.dir[k] = f.dir[k]; fs.center[k] = f.center[k]; }
        fs.scale = f.scale;
        fs.mode = f.type == "moment" ? 1 : (f.type == "totalPressure" ? 2 : (f.type == "massFlowRate" ? 3 : 0));
        fs.areaSum = 1.0;
        if (fs.mode == 2)
        {
            // areaSum_ of DAFunctionTotalPressure.C: total area of the function's faces, reduced over the ranks
            double a = 0.0;
            for (int p : f.patches)
                for (int i = 0; i < hm.patches[p].size; i++) a += hm.magSf[hm.patches[p].start + i];
            if (ghosted())
            {
                Solver* self = const_cast<Solver*>(this);
                if (self->dFacePart.n < 1) self->dFacePart.alloc(self->be, hm.nBF + 1);
                self->be.h2d(self->dFacePart.p, &a, sizeof(double));
                self->comm.allreduceSum(self->be, self->dFacePart.p, 1);
                self->be.d2h(&a, self->dFacePart.p, sizeof(double));
            }
            fs.areaSum = a;
        }
        if (f.type == "force" && f.dirMode != "fixedDirection")
        {
            // the angle of attack comes from the patchVelocity input (DAGlobalVar::patchVelocity, DAFunctionForce.C:92-114)
            const PatchVelocityDef& d = findPatchVelocity(f.patchVelocityInput);
            const double a = d.aoaDeg * 3.14159265358979323846 / 180.0;
            const double ca = std::cos(a), sa = std::sin(a);
            fs.dir[0] = fs.dir[1] = fs.dir[2] = 0.0;
            if (f.dirMode == "parallelToFlow")
            {
                fs.dir[d.flowAxis] = dAlpha ? -sa : ca;
                fs.dir[d.normalAxis] = dAlpha ? ca : sa;
            }
            else
            {
                fs.dir[d.flowAxis] = dAlpha ? -ca : -sa;
                fs.dir[d.normalAxis] = dAlpha ? -sa : ca;
            }
        }
        else if (dAlpha)
            fs.dir[0] = fs.dir[1] = fs.dir[2] = 0.0;
        return fs;
    }

    DevBuf<double> dFacePart;
    double gammaTPR = 1.4;
    int adjPCLag = 1; // > 1: solveLinearEqn keeps a preconditioner factorised at an earlier state
    bool keepPCMatrix = false; // writeJacobians lists dRdWTPC (or all): calcPC keeps the assembled values for export

    // dRdWTPC as assembled (rows: states, columns: residuals, both in the external numbering of this rank), CSR with sorted
    // columns -- what DAUtility::writeMatrixBinary(dRdWT, "dRdWTPC") stores (DASolver.C:1080-1085)
    void exportPC(std::vector<int64_t>& rowPtr, std::vector<int32_t>& cols, std::vector<double>& vals)
    {
        Krylov& K = kry;
        if (K.hValAssembled.size() != (size_t)K.ellSize || K.ellSize == 0)
            throw Error("the assembled dRdWTPC is not kept: list dRdWTPC in the writeJacobians option before calcdRdWT");
        std::vector<int32_t> hc((size_t)K.ellSize);
        be.d2h(hc.data(), K.dCol.p, (size_t)K.ellSize * sizeof(int32_t));
        rowPtr.assign((size_t)K.n + 1, 0);
        cols.clear();
        vals.clear();
        cols.reserve((size_t)K.nnz);
        vals.reserve((size_t)K.nnz);
        std::vector<std::pair<int32_t, double>> row;
        for (int e = 0; e < K.n; e++)
        {
            const int i = K.iperm[e];
            row.clear();
            for (int q = 0; q < K.rowLen[i]; q++)
            {
                const size_t at = (size_t)(K.rowBase[i] + (int64_t)q * K.rowStride[i]);
                row.emplace_back(K.perm[hc[at]], K.hValAssembled[at]);
            }
            std::sort(row.begin(), row.end());
            for (const auto& x : row)
            {
                cols.push_back(x.first);
                vals.push_back(x.second);
            }
            rowPtr[(size_t)e + 1] = (int64_t)cols.size();
        }
    }

    // the two area averages of DAFunctionTotalPressureRatio: side 0 = outlet (numerator), 1 = inlet
    ForceSpec tprSpec(const FunctionDef& f, int side) const
    {
        FunctionDef g = f;
        g.type = "totalPressure"; // the area sum of the side's patches
        g.patches = side == 0 ? f.outletPatches : f.inletPatches;
        g.scale = 1.0;
        ForceSpec fs = forceSpec(g);
        fs.mode = 4;
        fs.gamma = f.gamma;
        return fs;
    }
    double sumFaceParts(const ForceSpec& fs)
    {
        if (dFacePart.n < (size_t)hm.nBF + 1) dFacePart.alloc(be, hm.nBF + 1);
        if (par.comp) be.launch(hm.nBF, cForceFwd{mv, par, sv, rv, fs, dFacePart.p});
        else be.launch(hm.nBF, ForceFwd{mv, par, sv, rv, fs, dFacePart.p});
        std::vector<double> facePart(hm.nBF);
        be.d2h(facePart.data(), dFacePart.p, (size_t)hm.nBF * sizeof(double));
        double s = 0.0;
        for (int b = 0; b < hm.nBF; b++) s += facePart[b];
        if (ghosted())
        {
            be.h2d(dFacePart.p, &s, sizeof(double));
            comm.allreduceSum(be, dFacePart.p, 1);
            be.d2h(&s, dFacePart.p, sizeof(double));
        }
        return s;
    }
    // the face groups of a function with the weights of its derivative: F = sum_g (value of group g), or for the ratio
    // d(A/B) = dA/B - A/B^2 dB; `shift` makes the geometric derivative of the area averages exact (rev_kernels.hpp ForceSpec)
    std::vector<ForceSpec> derivativeSpecs(const FunctionDef& f)
    {
        std::vector<ForceSpec> out;
        if (f.type == "totalPressureRatio")
        {
            ForceSpec a = tprSpec(f, 0), b = tprSpec(f, 1);
            const double A = sumFaceParts(a), B = sumFaceParts(b);
            a.scale = 1.0 / B;
            a.shift = A;
            b.scale = -A / (B * B);
            b.shift = B;
            b.accumulate = 1;
            out.push_back(a);
            out.push_back(b);
            return out;
        }
        ForceSpec fs = forceSpec(f);
        if (fs.mode == 2) fs.shift = sumFaceParts(fs) / fs.scale;
        out.push_back(fs);
        return out;
    }

    double calcFunction(const std::string& name)
    {
        const FunctionDef& f = findFunction(name);
        ensureRecorded();
        if (f.type == "totalPressureRatio") return sumFaceParts(tprSpec(f, 0)) / sumFaceParts(tprSpec(f, 1));
        if (dFacePart.n < (size_t)hm.nBF + 1) dFacePart.alloc(be, hm.nBF + 1);
        if (par.comp) be.launch(hm.nBF, cForceFwd{mv, par, sv, rv, forceSpec(f), dFacePart.p});
        else be.launch(hm.nBF, ForceFwd{mv, par, sv, rv, forceSpec(f), dFacePart.p});
        std::vector<double> facePart(hm.nBF);
        be.d2h(facePart.data(), dFacePart.p, (size_t)hm.nBF * sizeof(double));
        // deterministic host summation in face order (the all-reduce of the reference, DAFunctionForce.C:146)
        double s = 0.0;
        for (int b = 0; b < hm.nBF; b++) s += facePart[b];
        if (ghosted())
        {
            be.h2d(dFacePart.p, &s, sizeof(double));
            comm.allreduceSum(be, dFacePart.p, 1);
            be.d2h(&s, dFacePart.p, sizeof(double));
        }
        return s;
    }

    // dF/d(|U|, aoa[deg]) at fixed states: only the flow-aligned direction modes depend on the angle
    void dFdPatchVelocity(const std::string& fname, double seed, double* product)
    {
        const FunctionDef& f = findFunction(fname);
        product[0] = product[1] = 0.0;
        if (f.type != "force" || f.dirMode == "fixedDirection") return;
        ensureRecorded();
        if (dFacePart.n < (size_t)hm.nBF + 1) dFacePart.alloc(be, hm.nBF + 1);
        ForceFwd k{mv, par, sv, rv, forceSpec(f, true), dFacePart.p};
        be.launch(hm.nBF, k);
        std::vector<double> facePart(hm.nBF);
        be.d2h(facePart.data(), dFacePart.p, (size_t)hm.nBF * sizeof(double));
        double s = 0.0;
        for (int b = 0; b < hm.nBF; b++) s += facePart[b];
        if (ghosted())
        {
            be.h2d(dFacePart.p, &s, sizeof(double));
            comm.allreduceSum(be, dFacePart.p, 1);
            be.d2h(&s, dFacePart.p, sizeof(double));
        }
        product[1] = seed * s * 3.14159265358979323846 / 180.0;
    }

    // [dF/dW]^T * seed, scaled by normalizeStates (DASolver.C:1819-1820)
    void dFdW(const std::string& name, double seed, double* out)
    {
        const FunctionDef& f = findFunction(name);
        ensureRecorded();
        if (par.comp)
        {
            std::vector<ForceSpec> specs;
            if (f.type == "totalPressureRatio") specs = derivativeSpecs(f);
            else specs.push_back(forceSpec(f));
            std::vector<double> part;
            for (size_t g = 0; g < specs.size(); g++)
            {
                be.zero(av.gPb, (size_t)3 * hm.nCtot * sizeof(double));
                be.zero(av.gNtb, (size_t)3 * hm.nCtot * sizeof(double));
                be.zero(av.gHeb, (size_t)3 * hm.nCtot * sizeof(double));
                launchNF<cForceRevA>(hm.nC, mv, par, sv, rv, av, specs[g], seed);
                if (ghosted()) halo.exchangeCells({{av.gUb, 9, 1, hm.nCtot}});
                launchNF<cRevC>(hm.nC, mv, par, sv, rv, av, dY2.p);
                be.zero(dY2.p + (size_t)nCellStates() * hm.nC, (size_t)hm.nF * sizeof(double)); // no face-flux dependence
                if (g == 0)
                    be.d2h(out, dY2.p, (size_t)nDof() * sizeof(double));
                else
                {
                    // the second face group of a ratio: the two sweeps add
                    part.resize(nDof());
                    be.d2h(part.data(), dY2.p, (size_t)nDof() * sizeof(double));
                    for (size_t i = 0; i < part.size(); i++) out[i] += part[i];
                }
            }
            return;
        }
        be.zero(av.gUb, (size_t)9 * hm.nCtot * sizeof(double));
        be.zero(av.gPb, (size_t)3 * hm.nCtot * sizeof(double));
        be.zero(av.gNtb, (size_t)3 * hm.nCtot * sizeof(double));
        launchNF<ForceRevA>(hm.nC, mv, par, sv, rv, av, forceSpec(f), seed);
        if (ghosted())
        {
            std::vector<HaloItem> it{{av.gUb, 9, 1, hm.nCtot}};
            halo.exchangeCells(it);
        }
        launchNF<RevC>(hm.nC, mv, par, sv, rv, av, dY2.p, 1);
        be.d2h(out, dY2.p, (size_t)nDof() * sizeof(double));
    }

    // ---- OpenFOAM field files (runTime.write() / DASolver::writeAdjointFields, DASolver.C:4055-4160) ---------------
    // ASCII vol/surface fields of a state-layout vector under <case>/<timeName>/<prefix><state>; one GPU
    void writeStateVector(const std::string& timeName, const std::string& prefix, const double* W) const
    {
        if (ghosted()) throw Error("field output needs an undecomposed mesh without cyclic patches in this build");
        const std::string dir = caseDirectory + "/" + timeName;
        ::mkdir(dir.c_str(), 0755);
        const int nC = hm.nC, nIF = hm.nIF;
        // stdio rather than iostreams: number formatting must not depend on the C++ locale machinery of the host process
        struct File
        {
            FILE* f;
            explicit File(const std::string& path) : f(fopen(path.c_str(), "w"))
            {
                if (!f) throw Error("cannot write " + path);
            }
            ~File() { fclose(f); }
        };
        auto header = [&](FILE* f, const char* cls, const std::string& name, const char* dims) {
            fprintf(f, "FoamFile\n{\n    version 2.0;\n    format ascii;\n    class %s;\n    location \"%s\";\n    object %s;\n}\n\n"
                       "dimensions %s;\n\n", cls, timeName.c_str(), name.c_str(), dims);
        };
        auto patches = [&](FILE* f, bool surface, const double* faceVals) {
            fprintf(f, "boundaryField\n{\n");
            for (size_t ip = 0; ip < hm.patches.size(); ip++)
            {
                const PatchDef& p = hm.patches[ip];
                fprintf(f, "    %s\n    {\n", p.name.c_str());
                if (surface)
                {
                    fprintf(f, "        type calculated;\n        value nonuniform List<scalar> %d(", p.size);
                    for (int i = 0; i < p.size; i++) fprintf(f, "%s%.17g", i ? " " : "", faceVals[p.start + i]);
                    fprintf(f, ");\n");
                }
                else
                    fprintf(f, "        type %s;\n", hm.patchGeom[ip] == PG_SYMMETRY ? "symmetry" : "zeroGradient");
                fprintf(f, "    }\n");
            }
            fprintf(f, "}\n");
        };
        {
            File o(dir + "/" + prefix + "U");
            header(o.f, "volVectorField", prefix + "U", "[0 1 -1 0 0 0 0]");
            fprintf(o.f, "internalField nonuniform List<vector> %d\n(\n", nC);
            for (int c = 0; c < nC; c++) fprintf(o.f, "(%.17g %.17g %.17g)\n", W[3 * c], W[3 * c + 1], W[3 * c + 2]);
            fprintf(o.f, ");\n\n");
            patches(o.f, false, nullptr);
        }
        std::vector<std::pair<std::string, const char*>> scal{{"p", par.comp ? "[1 -1 -2 0 0 0 0]" : "[0 2 -2 0 0 0 0]"}};
        if (par.comp) scal.push_back({"T", "[0 0 0 1 0 0 0]"});
        if (par.turb) scal.push_back({"nuTilda", "[0 2 -1 0 0 0 0]"});
        size_t off = (size_t)3 * nC;
        for (const auto& sc : scal)
        {
            File o(dir + "/" + prefix + sc.first);
            header(o.f, "volScalarField", prefix + sc.first, sc.second);
            fprintf(o.f, "internalField nonuniform List<scalar> %d\n(\n", nC);
            for (int c = 0; c < nC; c++) fprintf(o.f, "%.17g\n", W[off + c]);
            fprintf(o.f, ");\n\n");
            patches(o.f, false, nullptr);
            off += nC;
        }
        {
            File o(dir + "/" + prefix + "phi");
            header(o.f, "surfaceScalarField", prefix + "phi", par.comp ? "[1 0 -1 0 0 0 0]" : "[0 3 -1 0 0 0 0]");
            fprintf(o.f, "internalField nonuniform List<scalar> %d\n(\n", nIF);
            for (int i = 0; i < nIF; i++) fprintf(o.f, "%.17g\n", W[off + i]);
            fprintf(o.f, ");\n\n");
            patches(o.f, true, W + off);
        }
    }

    // writeSensMapField (DASolver.C:3962-4053): a cell field of derivatives as a dimensionless vol field <name> under <case>/<timeName>/,
    // boundary patches fixedValue zero
    void writeSensMapField(const std::string& name, const double* v, bool vector, const std::string& timeName) const
    {
        if (ghosted()) throw Error("field output needs an undecomposed mesh without cyclic patches in this build");
        const std::string dir = caseDirectory + "/" + timeName;
        ::mkdir(dir.c_str(), 0755);
        FILE* f = fopen((dir + "/" + name).c_str(), "w");
        if (!f) throw Error("cannot write " + dir + "/" + name);
        fprintf(f, "FoamFile\n{\n    version 2.0;\n    format ascii;\n    class %s;\n    location \"%s\";\n    object %s;\n}\n\n"
                   "dimensions [0 0 0 0 0 0 0];\n\n", vector ? "volVectorField" : "volScalarField", timeName.c_str(), name.c_str());
        fprintf(f, "internalField nonuniform List<%s> %d\n(\n", vector ? "vector" : "scalar", hm.nC);
        for (int c = 0; c < hm.nC; c++)
        {
            if (vector) fprintf(f, "(%.17g %.17g %.17g)\n", v[3 * c], v[3 * c + 1], v[3 * c + 2]);
            else fprintf(f, "%.17g\n", v[c]);
        }
        fprintf(f, ");\n\nboundaryField\n{\n");
        for (const PatchDef& p : hm.patches)
            fprintf(f, "    %s\n    {\n        type fixedValue;\n        value uniform %s;\n    }\n", p.name.c_str(), vector ? "(0 0 0)" : "0");
        fprintf(f, "}\n");
        fclose(f);
    }

    // writeSensMapSurface (DASolver.C:3840-3960): every point of every wall face takes the derivative of the closest design-surface
    // point; a face holds the sum over its points divided by 3 (the reference divides by vector::size(), not by the point count).
    // Returns the norm of the closest distances the reference prints.
    double writeSensMapSurface(const std::string& name, const double* dFdXs, const double* Xs, int size, const std::string& timeName) const
    {
        if (ghosted()) throw Error("field output needs an undecomposed mesh without cyclic patches in this build");
        const int nS = (int)std::lround(size / 3.0);
        if (nS <= 0) throw Error("writeSensMapSurface: empty surface");
        std::vector<double> sens((size_t)3 * hm.nBF, 0.0);
        double norm2 = 0.0;
        for (size_t ip = 0; ip < hm.patches.size(); ip++)
        {
            if (hm.patchGeom[ip] != PG_WALL) continue;
            const PatchDef& p = hm.patches[ip];
            for (int i = 0; i < p.size; i++)
            {
                const int f = p.start + i;
                for (int q = hm.fOff[f]; q < hm.fOff[f + 1]; q++)
                {
                    const int pt = hm.fLab[q];
                    double best = 9999999.0;
                    int bj = -1;
                    for (int j = 0; j < nS; j++)
                    {
                        double d2 = 0.0;
                        for (int k = 0; k < 3; k++) { const double d = Xs[3 * j + k] - hm.points[(size_t)3 * pt + k]; d2 += d * d; }
                        const double d = std::sqrt(d2);
                        if (d < best) { best = d; bj = j; }
                    }
                    if (bj < 0) throw Error("writeSensMapSurface: no surface point within 9999999 of a wall point");
                    norm2 += best * best;
                    for (int k = 0; k < 3; k++) sens[(size_t)3 * (f - hm.nIF) + k] += dFdXs[3 * bj + k];
                }
                for (int k = 0; k < 3; k++) sens[(size_t)3 * (f - hm.nIF) + k] /= 3.0;
            }
        }
        const std::string dir = caseDirectory + "/" + timeName;
        ::mkdir(dir.c_str(), 0755);
        FILE* f = fopen((dir + "/" + name).c_str(), "w");
        if (!f) throw Error("cannot write " + dir + "/" + name);
        fprintf(f, "FoamFile\n{\n    version 2.0;\n    format ascii;\n    class volVectorField;\n    location \"%s\";\n    object %s;\n}\n\n"
                   "dimensions [0 0 0 0 0 0 0];\n\ninternalField uniform (0 0 0);\n\nboundaryField\n{\n", timeName.c_str(), name.c_str());
        for (size_t ip = 0; ip < hm.patches.size(); ip++)
        {
            const PatchDef& p = hm.patches[ip];
            fprintf(f, "    %s\n    {\n        type fixedValue;\n", p.name.c_str());
            if (hm.patchGeom[ip] == PG_WALL)
            {
                fprintf(f, "        value nonuniform List<vector> %d(", p.size);
                for (int i = 0; i < p.size; i++)
                {
                    const double* v = &sens[(size_t)3 * (p.start + i - hm.nIF)];
                    fprintf(f, "%s(%.17g %.17g %.17g)", i ? " " : "", v[0], v[1], v[2]);
                }
                fprintf(f, ");\n");
            }
            else
                fprintf(f, "        value uniform (0 0 0);\n");
            fprintf(f, "    }\n");
        }
        fprintf(f, "}\n");
        fclose(f);
        return std::sqrt(norm2);
    }

    // writeMeshPoints (pyDASolvers.pyx:388-392) / writeCurrentMeshPointsToConstant / writeFailedMesh: <case>/<dirName>/polyMesh/points
    void writeMeshPoints(const double* pts, const std::string& dirName) const
    {
        if (ghosted()) throw Error("mesh output needs an undecomposed mesh without cyclic patches in this build");
        const std::string d1 = caseDirectory + "/" + dirName, d2 = d1 + "/polyMesh";
        ::mkdir(d1.c_str(), 0755);
        ::mkdir(d2.c_str(), 0755);
        FILE* f = fopen((d2 + "/points").c_str(), "w");
        if (!f) throw Error("cannot write " + d2 + "/points");
        fprintf(f, "FoamFile\n{\n    version 2.0;\n    format ascii;\n    class vectorField;\n    location \"%s/polyMesh\";\n    object points;\n}\n\n%d\n(\n",
                dirName.c_str(), hm.nP);
        for (int i = 0; i < hm.nP; i++) fprintf(f, "(%.17g %.17g %.17g)\n", pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]);
        fprintf(f, ")\n");
        fclose(f);
    }
    // readMeshPoints (pyDASolvers.pyx:385-386): the points written under a time directory become the mesh
    void readMeshPoints(const std::string& timeName)
    {
        std::vector<double> pts;
        readVectorField(caseDirectory + "/" + timeName + "/polyMesh/points", pts);
        if (pts.size() != hm.points.size()) throw Error("readMeshPoints: " + timeName + "/polyMesh/points has the wrong size");
        updateMesh(pts.data());
    }
    // readStateVars (pyDASolvers.pyx:382-383): the fields of a time directory become the states
    void readStateVars(const std::string& timeName) { initialStates(caseDirectory, timeName); }

    // ---- mesh coordinates as an input (volCoord) ------------------------------------------------------
    VolCoord volc;
    void uploadGeometry();
    void updateMesh(const double* pts);
    void volCoordSetup();
    void volCoordProduct(const double* psi, const FunctionDef* function, double seed, double* out);

    // ---- primal (SIMPLE) ----------------------------------------------------------------------------
    Primal primal;
    VecOps primalOps;
    void primalSetup();
    const double* primalSums(int k);
    void primalResidual(const EqnView& e, const double* x, const double* g, double* res);
    void primalJacobi(const EqnView& e, double* x, double* tmp, const double* g, const SegControl& ctl, double* res0);
    void primalCoarseSetup();
    void primalCoarseRefresh(const EqnView& e);
    void primalPrecond(const EqnView& e, const double* r, double* z);
    int primalPcg(const EqnView& e, double* x, const SegControl& ctl, double& res0);
    int solvePrimal(PrimalStats& st);

    // ---- Krylov -----------------------------------------------------------------------------------
    void pcSymbolic();
    void calcPC();
    void applyPC(const double* v, double* z);
    void applyIlu(const double* v, double* z);
    void coarseSetup();
    void coarseRestrict(const double* v, bool toHost = true);
    int kspExtraMatvecs = 0;
    int solveLinearEqn(const double* rhs, double* sol, KspStats& st);
    int solveIdrs(const double* rhs, double* sol, KspStats& st);
    int solveFixedPoint(const double* rhs, double* sol, KspStats& st);
};

} // namespace dab

#include "solver_krylov.hpp"
#include "solver_primal.hpp"
#include "solver_volcoord.hpp"
