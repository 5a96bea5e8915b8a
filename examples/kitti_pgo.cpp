// kitti_pgo.cpp -- the reference's two KITTI-00 Sim3 pose-graph pipelines on the B200 back-end.
//
//   direct    what testDirectSim3Optimization does   (kitti_surf.cpp:542-709)
//   stepwise  what testStepwiseSim3Optimization does (kitti_surf.cpp:713-1086): scale null-vector
//             initialisation -> 4-DoF scale+translation LM -> optional 7-DoF Sim3 LM
// written against include/sim3opt_b200/g2o_facade.hpp, i.e. with the reference's g2o spelling
// (SparseOptimizer, VertexSim3Expmap, EdgeSim3, OptimizationAlgorithmLevenberg(BlockSolverX(
// LinearSolverEigen))).  The graph is built exactly as the reference builds it: vertices in
// key-frame order, vertex 0 fixed, loop edges first, then the odometry edges, Omega = I.
//
// usage: kitti_pgo direct   <dataDir> <outFile> [--all-loops] [--iters N] [--numeric] [--pcg-tol T] [--precision P]
//                           [--marginals FILE]
//        kitti_pgo stepwise <dataDir> <outFile> [--all-loops] [--stages 2|3] [--no-stepwise] [--iters N] [--marginals FILE]
//        kitti_pgo online   <dataDir> <outFile> [--all-loops] [--step K] [--iters N] [--precision P]
//                           (key frames replayed one by one; grown with updateInitialization every K)
//        kitti_pgo dry-run  <dataDir> [--all-loops]        (no GPU: loads, builds, prints structure sizes)
//        kitti_pgo align    <resultFile> <gtPoseFile> [--only-scale]   (kitti_surf.cpp:1381-1452: Umeyama + RMSE)
//        kitti_pgo reproject <keyFrameDir> <resultFile> <out.bal>       (drawPTAMPoints.cpp:285-456: map -> BAL)
#define S3O_FACADE_EIGEN_NAMES
#include <chrono>
#include <cstring>
#include <iostream>
#include <map>

#include "sim3opt_b200/g2o_facade.hpp"
#include "sim3opt_b200/kitti_io.hpp"
#include "sim3opt_b200/map_io.hpp"

using namespace s3o::kitti;
using std::string;
using std::vector;

namespace {

struct Options {
    string mode, dataDir, outFile, marginalsFile;
    bool oneConstraint = true, stepwise = true, numeric = false;
    int stages = 2, iters = 100, precision = 6, step = 10;
    double pcgTol = 1e-13;
    int pcgMaxIter = 100000;
};

struct Timer {   // stands in for DUtils::Profiler (kitti_surf.cpp:546-547)
    std::map<string, double> ms;
    std::map<string, std::chrono::steady_clock::time_point> t0;
    void profile(const string &k) { t0[k] = std::chrono::steady_clock::now(); }
    void stop(const string &k) { ms[k] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0[k]).count(); }
};

g2o::OptimizationAlgorithmLevenberg *makeLevenberg() {
    std::unique_ptr<g2o::BlockSolverX::LinearSolverType> linearSolver =
        g2o::make_unique<g2o::LinearSolverEigen<g2o::BlockSolverX::PoseMatrixType>>();
    return new g2o::OptimizationAlgorithmLevenberg(g2o::make_unique<g2o::BlockSolverX>(std::move(linearSolver)));
}

// key frames + loop constraints with ids remapped from frame index to key-frame index
bool loadProblem(const Options &o, vector<KeyFrame> &kfs, vector<Sim3Constraint> &loops) {
    if (!GetAllKeyFrames(o.dataDir, kfs)) { std::cerr << "cannot read cc.txt / framePoses.txt in " << o.dataDir << "\n"; return false; }
    if (!LoadLoopConstraints(o.dataDir + "/loopConstraints.txt", loops) || loops.empty()) {
        std::cerr << "cannot read loopConstraints.txt in " << o.dataDir << "\n";
        return false;
    }
    if (o.oneConstraint) loops.resize(1, loops.front());
    std::map<int, int> frame2kf;
    for (const KeyFrame &kf : kfs) frame2kf[kf.mnId] = kf.mnFrameId;
    for (Sim3Constraint &c : loops) {
        auto a = frame2kf.find(c.trans_id1), b = frame2kf.find(c.trans_id2);
        if (a == frame2kf.end() || b == frame2kf.end()) { std::cerr << "loop constraint refers to a non-key frame\n"; return false; }
        c.trans_id1 = a->second;
        c.trans_id2 = b->second;
    }
    return true;
}

void configure(g2o::SparseOptimizer &opt, const Options &o) {
    opt.setAlgorithm(makeLevenberg());
    opt.setPcg(o.pcgTol, o.pcgMaxIter);
    if (o.numeric) opt.setJacobianMode(S3O_JAC_NUMERIC, 1e-9);   // g2o's linearizeOplus
}

void report(const char *stage, const g2o::SparseOptimizer &opt, int iters) {
    const vector<double> &h = opt.history();
    std::cout << stage << ": iterations " << iters << " free " << opt.numFreeVertices() << " blocks " << opt.numHessianBlocks();
    if (!h.empty()) std::cout << std::setprecision(12) << " chi2_first " << h[0] << " chi2_final " << h[h.size() - 5] << " lambda_final " << h[h.size() - 4];
    std::cout << "\n";
}

// Sim3 graph of both pipelines (kitti_surf.cpp:597-670 / :842-884)
void buildSim3Graph(g2o::SparseOptimizer &optimizer, const vector<KeyFrame> &kfs, const vector<Sim3Constraint> &loops,
                    const vector<g2o::Sim3> &vScw) {
    const Eigen::Matrix<double, 7, 7> matLambdasim = Eigen::Matrix<double, 7, 7>::Identity();
    for (const KeyFrame &kf : kfs) {
        vio::VertexSim3Expmap *vSim3 = new vio::VertexSim3Expmap();
        vSim3->setEstimate(vScw[kf.mnFrameId]);
        vSim3->setFixed(kf.mnFrameId == 0);
        vSim3->setId(kf.mnFrameId);
        vSim3->setMarginalized(false);
        optimizer.addVertex(vSim3);
    }
    for (const Sim3Constraint &c : loops) {
        vio::EdgeSim3 *esim = new vio::EdgeSim3();
        esim->setVertex(1, optimizer.vertex(c.trans_id2));
        esim->setVertex(0, optimizer.vertex(c.trans_id1));
        esim->setMeasurement(c.mean);
        esim->information() = matLambdasim;
        optimizer.addEdge(esim);
    }
    for (size_t i = 1; i < kfs.size(); ++i) {      // spanning-tree (odometry) edges
        const int nIDi = kfs[i].mnFrameId, nIDj = kfs[i - 1].mnFrameId;
        const g2o::Sim3 Sji = vScw[nIDj] * vScw[nIDi].inverse();
        vio::EdgeSim3 *e = new vio::EdgeSim3();
        e->setVertex(1, optimizer.vertex(nIDj));
        e->setVertex(0, optimizer.vertex(nIDi));
        e->setMeasurement(Sji);
        e->information() = matLambdasim;
        optimizer.addEdge(e);
    }
}

// --marginals FILE: the d x d block of H^-1 at the final estimates (g2o computeMarginals) of every free key frame,
// one line each: key-frame id, then the block row by row
bool writeMarginals(const Options &o, const vector<KeyFrame> &kfs, g2o::SparseOptimizer &opt, int d) {
    if (o.marginalsFile.empty()) return true;
    g2o::SparseOptimizer::VertexContainer freeVertices;
    for (const KeyFrame &kf : kfs)
        if (!opt.vertex(kf.mnFrameId)->fixed()) freeVertices.push_back(opt.vertex(kf.mnFrameId));
    g2o::SparseBlockMatrix<g2o::MatrixX> spinv;
    if (!opt.computeMarginals(spinv, freeVertices)) { std::cerr << "computeMarginals: " << opt.lastError() << "\n"; return false; }
    FILE *f = std::fopen(o.marginalsFile.c_str(), "w");
    if (!f) { std::cerr << "cannot write " << o.marginalsFile << "\n"; return false; }
    std::fprintf(f, "%% marginal covariance of each free key frame: kf id, %dx%d block of H^-1 (row-major)\n", d, d);
    for (const KeyFrame &kf : kfs) {
        const g2o::Vertex *v = opt.vertex(kf.mnFrameId);
        if (v->fixed()) continue;
        const g2o::MatrixX *b = spinv.block(v->hessianIndex(), v->hessianIndex());
        std::fprintf(f, "%d", kf.mnId);
        for (int k = 0; k < d * d; ++k) std::fprintf(f, " %.17g", b->data()[k]);
        std::fprintf(f, "\n");
    }
    std::fclose(f);
    std::cout << "saved marginals file " << o.marginalsFile << "\n";
    return true;
}

template <class GetSim3>
void writeResult(const Options &o, const vector<KeyFrame> &kfs, const char *header, GetSim3 get) {
    std::ofstream log(o.outFile);
    log << header << "\n";
    for (const KeyFrame &kf : kfs) WriteSim3Line(log, kf.mnId, get(kf.mnFrameId), o.precision);
    std::cout << "saved output file " << o.outFile << "\n";
}

int runDirect(const Options &o) {
    Timer profiler;
    profiler.profile("sim3_direct");
    vector<KeyFrame> kfs;
    vector<Sim3Constraint> loops;
    if (!loadProblem(o, kfs, loops)) return 2;
    g2o::SparseOptimizer optimizer;
    configure(optimizer, o);
    vector<g2o::Sim3> vScw(kfs.size());
    for (const KeyFrame &kf : kfs) vScw[kf.mnFrameId] = g2o::Sim3(kf.GetRotation(), kf.GetTranslation(), 1.0);
    buildSim3Graph(optimizer, kfs, loops, vScw);
    if (o.mode == "dry-run") {
        // host-only twin of the structure build: sizes without touching a GPU
        const int n = (int)kfs.size(), ne = (int)optimizer.edges().size();
        vector<uint8_t> fixed(n, 0);
        fixed[0] = 1;
        vector<int32_t> v0(ne), v1(ne), colptr(n + 1), rowidx(n + ne);
        for (int k = 0; k < ne; ++k) { v0[k] = optimizer.edges()[k]->vertex(0)->id(); v1[k] = optimizer.edges()[k]->vertex(1)->id(); }
        int nf = 0, nb = 0;
        if (s3o_host_structure(n, fixed.data(), ne, v0.data(), v1.data(), &nf, &nb, colptr.data(), rowidx.data(), nullptr) != S3O_OK) {
            std::cerr << s3o_last_error() << "\n";
            return 3;
        }
        std::cout << "dry-run: vertices " << n << " edges " << ne << " free " << nf << " blocks " << nb << "\n";
        return 0;
    }
    if (!optimizer.initializeOptimization()) { std::cerr << "initializeOptimization: " << optimizer.lastError() << "\n"; return 3; }
    profiler.profile("optimize");
    const int iters = optimizer.optimize(o.iters);
    profiler.stop("optimize");
    if (iters <= 0) { std::cerr << "optimize: " << optimizer.lastError() << "\n"; return 3; }
    report("direct", optimizer, iters);
    if (!writeMarginals(o, kfs, optimizer, 7)) return 3;
    writeResult(o, kfs, "% sim3 optimization result: kf id, sw2i, scaled tiinw, ri2w(qxyzw):", [&](int id) {
        return static_cast<vio::VertexSim3Expmap *>(optimizer.vertex(id))->estimate();
    });
    profiler.stop("sim3_direct");
    std::cout << "Execution time:\n sim3 direct optimization: " << profiler.ms["sim3_direct"] << " ms (optimize " << profiler.ms["optimize"] << " ms)\n";
    return 0;
}

// online: the key frames replayed one by one, as a SLAM back-end receives them.  Step k adds key frame k, its
// odometry edge (k, k-1) and every loop edge whose two key frames now exist; every --step K key frames the graph is
// grown on the device (updateInitialization) and optimised with optimize(--iters, true).
int runOnline(const Options &o) {
    vector<KeyFrame> kfs;
    vector<Sim3Constraint> loops;
    if (!loadProblem(o, kfs, loops)) return 2;
    g2o::SparseOptimizer optimizer;
    configure(optimizer, o);
    const Eigen::Matrix<double, 7, 7> matLambdasim = Eigen::Matrix<double, 7, 7>::Identity();
    vector<g2o::Sim3> vScw(kfs.size());
    for (const KeyFrame &kf : kfs) vScw[kf.mnFrameId] = g2o::Sim3(kf.GetRotation(), kf.GetTranslation(), 1.0);
    g2o::HyperGraph::VertexSet vset;
    g2o::HyperGraph::EdgeSet eset;
    auto edge = [&](int id0, int id1, const g2o::Sim3 &m) {
        vio::EdgeSim3 *e = new vio::EdgeSim3();
        e->setVertex(1, optimizer.vertex(id1));
        e->setVertex(0, optimizer.vertex(id0));
        e->setMeasurement(m);
        e->information() = matLambdasim;
        optimizer.addEdge(e);
        eset.insert(e);
    };
    Timer profiler;
    bool initialised = false;
    int merges = 0, total_iters = 0;
    for (size_t k = 0; k < kfs.size(); ++k) {
        const int id = kfs[k].mnFrameId;
        vio::VertexSim3Expmap *v = new vio::VertexSim3Expmap();
        v->setEstimate(vScw[id]);
        v->setFixed(id == 0);
        v->setId(id);
        optimizer.addVertex(v);
        vset.insert(v);
        if (k > 0) edge(id, kfs[k - 1].mnFrameId, vScw[kfs[k - 1].mnFrameId] * vScw[id].inverse());
        for (const Sim3Constraint &c : loops)
            if (std::max(c.trans_id1, c.trans_id2) == id) edge(c.trans_id1, c.trans_id2, c.mean);
        if ((k + 1) % o.step != 0 && k + 1 != kfs.size()) continue;
        profiler.profile("grow");
        const bool ok = initialised ? optimizer.updateInitialization(vset, eset) : optimizer.initializeOptimization();
        profiler.stop("grow");
        if (!ok) { std::cerr << "update / initialize: " << optimizer.lastError() << "\n"; return 3; }
        initialised = true;
        vset.clear();
        eset.clear();
        profiler.profile("optimize");
        const int iters = optimizer.optimize(o.iters, true);
        profiler.stop("optimize");
        if (iters < 0) { std::cerr << "optimize: " << optimizer.lastError() << "\n"; return 3; }
        total_iters += iters;
        ++merges;
    }
    report("online", optimizer, total_iters);
    std::cout << "online: merges " << merges << " grow " << profiler.ms["grow"] << " ms optimize " << profiler.ms["optimize"] << " ms\n";
    writeResult(o, kfs, "% sim3 optimization result: kf id, sw2i, scaled tiinw, ri2w(qxyzw):", [&](int id) {
        return static_cast<vio::VertexSim3Expmap *>(optimizer.vertex(id))->estimate();
    });
    return 0;
}

// Scale initialisation of the stepwise pipeline (kitti_surf.cpp:887-934).  The reference takes the
// right singular vector of the smallest singular value of the (N-1+L) x N matrix with rows
// x[k-1] - x[k] (odometry) and s_loop x[id1] - x[id2] (loops) by a dense Jacobi SVD.  That matrix
// is the Jacobian of the 1-DoF scale graph with no vertex fixed, so its Gram matrix is that graph's
// Hessian: the same vector is the eigenvector of the smallest eigenvalue, found on the device by
// inverse iteration with the PCG solver (s3o_smallest_eigenvector).
bool solveScalesByNullVector(const Options &o, const vector<KeyFrame> &kfs, const vector<Sim3Constraint> &loops,
                             const vector<g2o::Sim3> &vScw, vector<double> &allScales) {
    const int n = (int)kfs.size();
    vector<double> est(n, 1.0), meas;
    vector<int32_t> v0, v1;
    for (const Sim3Constraint &c : loops) { v0.push_back(c.trans_id1); v1.push_back(c.trans_id2); meas.push_back(c.mean.scale()); }
    for (int i = 1; i < n; ++i) { v0.push_back(i); v1.push_back(i - 1); meas.push_back((vScw[i - 1] * vScw[i].inverse()).scale()); }
    s3o_problem *p = nullptr;
    if (s3o_create(S3O_KIND_SCALE, 0, &p) != S3O_OK) return false;
    bool ok = s3o_set_vertices(p, n, est.data(), nullptr, nullptr) == S3O_OK &&
              s3o_set_edges(p, (int)v0.size(), v0.data(), v1.data(), meas.data(), nullptr) == S3O_OK &&
              s3o_set_pcg(p, 1e-12, 100000) == S3O_OK;
    double smin = 0, smax = 0;
    int its = 0;
    allScales.assign(n, 0.0);
    ok = ok && s3o_smallest_eigenvector(p, 50, 1e-12, allScales.data(), &smin, &smax, &its) == S3O_OK;
    if (!ok) std::cerr << "scale null vector: " << s3o_last_error() << "\n";
    s3o_destroy(p);
    if (!ok) return false;
    if (std::sqrt(smax) * 5e-4 > std::sqrt(smin)) std::cout << "Warning possible unsable result by SVD\n";
    const double first = allScales[0];
    for (double &s : allScales) s /= first;
    std::cout << "scale_dlt: inverse iterations " << its << " sigma_min " << std::sqrt(smin) << " sigma_max " << std::sqrt(smax) << "\n";
    (void)o;
    return true;
}

int runStepwise(const Options &o) {
    Timer profiler;
    profiler.profile("tot_optim");
    const int num_optimizer = o.stepwise ? o.stages : 3;
    vector<KeyFrame> kfs;
    vector<Sim3Constraint> loops;
    if (!loadProblem(o, kfs, loops)) return 2;
    // optimizer[1]: 4-DoF scale+translation; optimizer[2]: 7-DoF Sim3.  (The reference also fills a
    // 1-DoF optimizer[0] but never optimises it, kitti_surf.cpp:938-960.)
    g2o::SparseOptimizer optimizerST, optimizerSim3;
    configure(optimizerST, o);
    configure(optimizerSim3, o);
    const Eigen::Matrix<double, 4, 4> matLambdast = Eigen::Matrix<double, 4, 4>::Identity();
    vector<g2o::Sim3> vScw(kfs.size());
    for (const KeyFrame &kf : kfs) {
        const int nIDi = kf.mnFrameId;
        const Eigen::Matrix3d Rcw = kf.GetRotation();
        const g2o::Sim3 Siw(Rcw, kf.GetTranslation(), 1.0);
        vScw[nIDi] = Siw;
        vio::G2oVertexScaleTrans *vST = new vio::G2oVertexScaleTrans();
        vST->setEstimate(toScaleTrans(Siw));
        vST->Rw2i = vio::SO3(Rcw);
        vST->setFixed(nIDi == 0);
        vST->setId(nIDi);
        vST->setMarginalized(false);
        optimizerST.addVertex(vST);
    }
    auto addST = [&](int idI, int idJ, const g2o::Sim3 &Sji) {
        vio::G2oEdgeScaleTrans *est = new vio::G2oEdgeScaleTrans();
        est->setVertex(1, optimizerST.vertex(idJ));
        est->setVertex(0, optimizerST.vertex(idI));
        est->setMeasurement(toScaleTrans(Sji));
        est->information() = matLambdast;
        optimizerST.addEdge(est);
    };
    for (const Sim3Constraint &c : loops) addST(c.trans_id1, c.trans_id2, c.mean);
    for (size_t i = 1; i < kfs.size(); ++i) addST((int)i, (int)i - 1, vScw[i - 1] * vScw[i].inverse());
    if (num_optimizer == 3) buildSim3Graph(optimizerSim3, kfs, loops, vScw);

    if (o.stepwise) {
        profiler.profile("scale_dlt");
        vector<double> allScales;
        if (!solveScalesByNullVector(o, kfs, loops, vScw, allScales)) return 3;
        for (const KeyFrame &kf : kfs) {
            vio::G2oVertexScaleTrans *vST = static_cast<vio::G2oVertexScaleTrans *>(optimizerST.vertex(kf.mnFrameId));
            Eigen::Vector4d stw2i = vST->estimate();
            stw2i[0] = allScales[kf.mnFrameId];
            vST->setEstimate(stw2i);
        }
        profiler.stop("scale_dlt");
        profiler.profile("scale_trans");
        if (!optimizerST.initializeOptimization()) { std::cerr << optimizerST.lastError() << "\n"; return 3; }
        const int it = optimizerST.optimize(o.iters);
        profiler.stop("scale_trans");
        if (it <= 0) { std::cerr << "scale_trans optimize: " << optimizerST.lastError() << "\n"; return 3; }
        report("scale_trans", optimizerST, it);
        if (num_optimizer != 3 && !writeMarginals(o, kfs, optimizerST, 4)) return 3;
    }
    auto stToSim3 = [&](int id) {
        vio::G2oVertexScaleTrans *vST = static_cast<vio::G2oVertexScaleTrans *>(optimizerST.vertex(id));
        const Eigen::Vector4d stw2i = vST->estimate();
        return g2o::Sim3(vST->Rw2i.unit_quaternion(), Eigen::Vector3d(stw2i.tail<3>()), stw2i[0]);
    };
    if (num_optimizer == 3) {
        for (const KeyFrame &kf : kfs)
            static_cast<vio::VertexSim3Expmap *>(optimizerSim3.vertex(kf.mnFrameId))->setEstimate(stToSim3(kf.mnFrameId));
        profiler.profile("sim3_optim");
        if (!optimizerSim3.initializeOptimization()) { std::cerr << optimizerSim3.lastError() << "\n"; return 3; }
        const int it = optimizerSim3.optimize(o.iters);
        profiler.stop("sim3_optim");
        if (it <= 0) { std::cerr << "sim3 optimize: " << optimizerSim3.lastError() << "\n"; return 3; }
        report("sim3_optim", optimizerSim3, it);
        if (!writeMarginals(o, kfs, optimizerSim3, 7)) return 3;
    }
    writeResult(o, kfs, "% sim3 optimization result: kf frameid, sw2i, scaled tiinw, ri2w(qxyzw):", [&](int id) {
        return num_optimizer == 3 ? static_cast<vio::VertexSim3Expmap *>(optimizerSim3.vertex(id))->estimate() : stToSim3(id);
    });
    profiler.stop("tot_optim");
    std::cout << "Execution time:\n total optimization: " << profiler.ms["tot_optim"] << " ms\n scale dlt: " << profiler.ms["scale_dlt"]
              << " ms\n scale_trans: " << profiler.ms["scale_trans"] << " ms\n sim3_optim: " << profiler.ms["sim3_optim"] << " ms\n";
    return 0;
}

// ALIGN_TRAJECTORIES_OPTIMIZED (kitti_surf.cpp:1381-1452): similarity-align an optimised key-frame
// trajectory to the KITTI ground truth and report RMSE / max deviation / their ratio to the path length.
int runAlign(const string &resultFile, const string &gtFile, bool onlyScale) {
    vector<g2o::Vector3> gt, opt;
    vector<int> ids;
    if (!ReadKITTIPosePositions(gtFile, gt)) { std::cerr << "cannot read " << gtFile << "\n"; return 2; }
    if (!ReadOptimizedSim3Positions(resultFile, ids, opt)) { std::cerr << "cannot read " << resultFile << "\n"; return 2; }
    std::cout << "Num of lines:" << gt.size() << "\nNum of lines:" << opt.size() << "\n";
    double totalDistance = 0;
    for (size_t j = 1; j < gt.size(); ++j) totalDistance += (gt[j] - gt[j - 1]).norm();
    vector<double> q, t;
    for (size_t j = 0; j < ids.size(); ++j) {
        if (ids[j] < 0 || ids[j] >= (int)gt.size()) { std::cerr << "frame id " << ids[j] << " not in the ground truth\n"; return 2; }
        for (int c = 0; c < 3; ++c) { q.push_back(opt[j][c]); t.push_back(gt[ids[j]][c]); }
    }
    double S221[16], rmse = 0, maxError = 0;
    if (s3o_align_similarity(0, (int)ids.size(), q.data(), t.data(), onlyScale ? 1 : 0, S221, &rmse, &maxError) != S3O_OK) {
        std::cerr << s3o_last_error() << "\n";
        return 3;
    }
    std::cout << "estimated similarity transform by umeyama \n";
    std::cout.precision(9);
    for (int r = 0; r < 4; ++r) std::cout << S221[r * 4] << " " << S221[r * 4 + 1] << " " << S221[r * 4 + 2] << " " << S221[r * 4 + 3] << "\n";
    std::cout << "RMSE and Max deviation " << rmse << " " << maxError << "\n";
    std::cout << "total distance " << totalDistance << " ratio of rmse and max error " << rmse / totalDistance << " "
              << maxError / totalDistance << "\n";
    return 0;
}

// figureKITTIBA (drawPTAMPoints.cpp:285-456, called at kitti_surf.cpp:1337,1375): key-frame dumps + optimised
// trajectory -> BAL file for ba_demo.  S221 is the identity here, as at the reference's call sites.
int runReproject(const string &keyFrameDir, const string &resultFile, const string &balFile) {
    s3o::mapio::BalProblem P;
    string err;
    if (!s3o::mapio::ReprojectMap(keyFrameDir, resultFile, RobotVision::Sim3<>(), P, &err)) { std::cerr << err << "\n"; return 2; }
    if (!s3o::mapio::SaveBALFile(P, balFile)) { std::cerr << "cannot write " << balFile << "\n"; return 2; }
    std::cout << "cameras " << P.Rw2c.size() << " points " << P.points.size() << " observations " << P.obs.size() << "\n";
    std::cout << "saved output file " << balFile << "\n";
    return 0;
}

}  // namespace

int main(int argc, char **argv) {
    Options o;
    if (argc < 3) {
        std::cerr << "usage: kitti_pgo direct|stepwise|online|dry-run <dataDir> [<outFile>] [--all-loops] [--stages 2|3] [--no-stepwise] [--step K]"
                     " [--iters N] [--numeric] [--pcg-tol T] [--precision P] [--marginals FILE]\n";
        return 1;
    }
    o.mode = argv[1];
    o.dataDir = argv[2];
    if (o.mode == "align") {       // kitti_pgo align <resultFile> <gtPoseFile> [--only-scale]
        if (argc < 4) { std::cerr << "usage: kitti_pgo align <resultFile> <gtPoseFile> [--only-scale]\n"; return 1; }
        return runAlign(argv[2], argv[3], argc > 4 && string(argv[4]) == "--only-scale");
    }
    if (o.mode == "reproject") {   // kitti_pgo reproject <keyFrameDir> <resultFile> <out.bal>
        if (argc < 5) { std::cerr << "usage: kitti_pgo reproject <keyFrameDir> <resultFile> <out.bal>\n"; return 1; }
        return runReproject(argv[2], argv[3], argv[4]);
    }
    int k = 3;
    if (o.mode != "dry-run") {
        if (argc < 4) { std::cerr << "missing <outFile>\n"; return 1; }
        o.outFile = argv[3];
        k = 4;
    }
    for (; k < argc; ++k) {
        const string a = argv[k];
        if (a == "--all-loops") o.oneConstraint = false;
        else if (a == "--no-stepwise") o.stepwise = false;
        else if (a == "--numeric") o.numeric = true;
        else if (a == "--stages" && k + 1 < argc) o.stages = std::atoi(argv[++k]);
        else if (a == "--iters" && k + 1 < argc) o.iters = std::atoi(argv[++k]);
        else if (a == "--step" && k + 1 < argc) o.step = std::max(1, std::atoi(argv[++k]));
        else if (a == "--precision" && k + 1 < argc) o.precision = std::atoi(argv[++k]);
        else if (a == "--pcg-tol" && k + 1 < argc) o.pcgTol = std::atof(argv[++k]);
        else if (a == "--marginals" && k + 1 < argc) o.marginalsFile = argv[++k];
        else { std::cerr << "unknown option " << a << "\n"; return 1; }
    }
    if (o.mode != "dry-run") {
        // One-time cost of the process, not of the optimisation: creating the CUDA context and loading the kernels
        // (about a second on a fresh process).  Paid here, reported on its own line, so that the reference's timers
        // (kitti_surf.cpp:705-708, :1079-1085) measure the pipeline stages only.
        const auto t0 = std::chrono::steady_clock::now();
        s3o_problem *warm = nullptr;
        if (s3o_create(S3O_KIND_SCALE, 0, &warm) != S3O_OK) { std::cerr << s3o_last_error() << "\n"; return 3; }
        s3o_destroy(warm);
        std::cout << "cuda context: " << std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() << " ms\n";
    }
    if (o.mode == "direct" || o.mode == "dry-run") return runDirect(o);
    if (o.mode == "stepwise") return runStepwise(o);
    if (o.mode == "online") return runOnline(o);
    std::cerr << "unknown mode " << o.mode << "\n";
    return 1;
}
