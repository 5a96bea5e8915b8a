// g2o_facade.hpp -- the reference's graph-construction / optimiser API over the sim3opt_b200 C ABI.
//
// The reference drives its hot path through g2o (SURVEY.md section 8b):
//     g2o::SparseOptimizer optimizer;                                   kitti_surf.cpp:552
//     auto linearSolver = g2o::make_unique<g2o::LinearSolverEigen<...>>();          :553-554
//     auto* solver = new g2o::OptimizationAlgorithmLevenberg(
//                        g2o::make_unique<g2o::BlockSolverX>(std::move(linearSolver)));  :556-557
//     optimizer.setAlgorithm(solver);                                               :558
//     v = new vio::VertexSim3Expmap(); v->setEstimate(Siw); v->setFixed(..); v->setId(..);
//     optimizer.addVertex(v);                                                       :602-620
//     e = new vio::EdgeSim3(); e->setVertex(0|1, ..); e->setMeasurement(..);
//     e->information() = I7; optimizer.addEdge(e);                                  :633-638
//     optimizer.initializeOptimization(); optimizer.optimize(100);                  :674-675
//     static_cast<vio::VertexSim3Expmap*>(optimizer.vertex(id))->estimate();        :688-689
// This header keeps those names, argument meanings and return conventions (namespaces g2o:: and
// vio::).  The classes only RECORD the graph in host memory; initializeOptimization() flattens it
// into arrays and hands it to the C ABI (include/sim3opt_b200.h), optimize() runs the whole
// Levenberg-Marquardt loop on the GPU and copies the estimates back into the vertex objects.
// The "linear solver" objects are plugin-slot placeholders: the cut is at the OptimizationAlgorithm
// level, so H, b and x never leave the device.  There is no CPU path: without a CUDA device
// initializeOptimization() returns false and optimize() returns -1 (lastError() has the reason).
//
// Ownership follows g2o: vertices, edges, robust kernels and parameters are new-ed by the caller
// and owned by the graph after addVertex/addEdge; the algorithm is owned after setAlgorithm.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "../sim3opt_b200.h"
#include "linalg.hpp"

namespace g2o {

using s3o::Matrix;
using Matrix3 = s3o::Matrix<double, 3, 3>;
using Vector3 = s3o::Matrix<double, 3, 1>;
using Vector4 = s3o::Matrix<double, 4, 1>;
using Vector7 = s3o::Matrix<double, 7, 1>;
using Quaternion = s3o::Quaternion<double>;

template <class T, class... Args>
std::unique_ptr<T> make_unique(Args &&...args) { return std::unique_ptr<T>(new T(std::forward<Args>(args)...)); }

// ---- g2o::Sim3 (row a8): x -> s (r x) + t ------------------------------------------------------
class Sim3 {
public:
    Sim3() : s_(1.0) {}
    Sim3(const Quaternion &r, const Vector3 &t, double s) : r_(r), t_(t), s_(s) { r_.normalize(); }
    Sim3(const Matrix3 &R, const Vector3 &t, double s) : r_(R), t_(t), s_(s) {}
    const Quaternion &rotation() const { return r_; }
    const Vector3 &translation() const { return t_; }
    double scale() const { return s_; }
    void setRotation(const Quaternion &r) { r_ = r; }
    void setTranslation(const Vector3 &t) { t_ = t; }
    void setScale(double s) { s_ = s; }
    Vector3 map(const Vector3 &xyz) const { return (r_ * xyz) * s_ + t_; }
    Sim3 inverse() const {
        const Quaternion ri = r_.conjugate();
        return Sim3(ri, ri * (t_ * (-1.0 / s_)), 1.0 / s_);
    }
    Sim3 operator*(const Sim3 &o) const { return Sim3(r_ * o.r_, (r_ * o.t_) * s_ + t_, s_ * o.s_); }
    Sim3 &operator*=(const Sim3 &o) { *this = *this * o; return *this; }
    // C-ABI state layout [qx qy qz qw tx ty tz s]
    void pack(double *x) const {
        x[0] = r_.x(); x[1] = r_.y(); x[2] = r_.z(); x[3] = r_.w();
        x[4] = t_[0]; x[5] = t_[1]; x[6] = t_[2]; x[7] = s_;
    }
    static Sim3 unpack(const double *x) {
        Sim3 S;
        S.r_ = Quaternion(x[3], x[0], x[1], x[2]);
        S.t_ = Vector3(x[4], x[5], x[6]);
        S.s_ = x[7];
        return S;
    }

private:
    Quaternion r_;
    Vector3 t_;
    double s_;
};

// ---- g2o::MatrixX and g2o::SparseBlockMatrix<MatrixX>: what computeMarginals fills -------------------------
class MatrixX {      // dense, row-major
public:
    MatrixX() {}
    MatrixX(int rows, int cols) : rows_(rows), cols_(cols), data_((size_t)rows * cols, 0.0) {}
    int rows() const { return rows_; }
    int cols() const { return cols_; }
    double &operator()(int r, int c) { return data_[(size_t)r * cols_ + c]; }
    double operator()(int r, int c) const { return data_[(size_t)r * cols_ + c]; }
    double *data() { return data_.data(); }
    const double *data() const { return data_.data(); }

private:
    int rows_ = 0, cols_ = 0;
    std::vector<double> data_;
};

template <class MatrixType>
class SparseBlockMatrix {
public:
    SparseBlockMatrix() {}
    // rbi / cbi: the cumulative row / column index at the end of each block row / column, as in g2o
    SparseBlockMatrix(const int *rbi, const int *cbi, int rb, int cb, bool /*hasStorage*/ = true)
        : rbi_(rbi, rbi + rb), cbi_(cbi, cbi + cb) {}
    // block (r, c), or nullptr when it is not stored; alloc = true creates a zero block
    MatrixType *block(int r, int c, bool alloc = false) {
        auto it = blocks_.find({ r, c });
        if (it != blocks_.end()) return &it->second;
        if (!alloc || r < 0 || c < 0 || r >= (int)rbi_.size() || c >= (int)cbi_.size()) return nullptr;
        return &blocks_.emplace(std::make_pair(r, c), MatrixType(rowsOfBlock(r), colsOfBlock(c))).first->second;
    }
    const MatrixType *block(int r, int c) const {
        auto it = blocks_.find({ r, c });
        return it == blocks_.end() ? nullptr : &it->second;
    }
    int rowsOfBlock(int r) const { return r ? rbi_[r] - rbi_[r - 1] : rbi_[0]; }
    int colsOfBlock(int c) const { return c ? cbi_[c] - cbi_[c - 1] : cbi_[0]; }
    int rowBaseOfBlock(int r) const { return r ? rbi_[r - 1] : 0; }
    int colBaseOfBlock(int c) const { return c ? cbi_[c - 1] : 0; }
    const std::vector<int> &rowBlockIndices() const { return rbi_; }
    const std::vector<int> &colBlockIndices() const { return cbi_; }

private:
    std::vector<int> rbi_, cbi_;
    std::map<std::pair<int, int>, MatrixType> blocks_;
};

// ---- robust kernels (row a13) ------------------------------------------------------------------
class RobustKernel {
public:
    virtual ~RobustKernel() {}
    virtual void setDelta(double d) { delta_ = d; }
    double delta() const { return delta_; }
    virtual int s3oKind() const = 0;

protected:
    double delta_ = 1.0;
};
class RobustKernelHuber : public RobustKernel {
public:
    int s3oKind() const override { return S3O_ROBUST_HUBER; }
};

// ---- vertices and edges ------------------------------------------------------------------------
class SparseOptimizer;

class Vertex {   // HyperGraph::Vertex + OptimizableGraph::Vertex, the members the reference touches
public:
    virtual ~Vertex() {}
    int id() const { return id_; }
    void setId(int id) { id_ = id; }
    bool fixed() const { return fixed_; }
    void setFixed(bool f) { fixed_ = f; }
    bool marginalized() const { return marginalized_; }
    void setMarginalized(bool m) { marginalized_ = m; }
    int hessianIndex() const { return hessian_index_; }
    virtual int dimension() const = 0;          // minimal (tangent) dimension
    virtual int estimateDimension() const = 0;  // doubles of the C-ABI state
    virtual int s3oKind() const = 0;
    virtual void packEstimate(double *x) const = 0;
    virtual void unpackEstimate(const double *x) = 0;
    virtual bool packAux(double * /*q4*/) const { return false; }
    virtual int baRole() const { return -1; }   // kind BA only: 0 = camera (pose), 1 = point (landmark)

private:
    friend class SparseOptimizer;
    int id_ = -1, hessian_index_ = -1;
    bool fixed_ = false, marginalized_ = false;
};

template <int D, class T>
class BaseVertex : public Vertex {
public:
    static const int Dimension = D;
    typedef T EstimateType;
    const T &estimate() const { return estimate_; }
    void setEstimate(const T &e) { estimate_ = e; }
    int dimension() const override { return D; }

protected:
    T estimate_;
};

class Edge {   // OptimizableGraph::Edge
public:
    virtual ~Edge() { delete robust_; }
    void setVertex(size_t i, Vertex *v) { if (i < 2) v_[i] = v; }
    Vertex *vertex(size_t i) const { return i < 2 ? v_[i] : nullptr; }
    void setRobustKernel(RobustKernel *k) { delete robust_; robust_ = k; }   // owned, as in g2o
    RobustKernel *robustKernel() const { return robust_; }
    bool setParameterId(int /*argNum*/, int paramId) { param_id_ = paramId; return true; }
    int parameterId() const { return param_id_; }
    virtual int dimension() const = 0;
    virtual int s3oKind() const = 0;
    virtual void packMeasurement(double *m) const = 0;
    virtual void packInformation(double *info /* D*D row-major */) const = 0;
    virtual bool informationIsIdentity() const = 0;
    virtual void unpackError(const double *e) = 0;
    virtual double chi2() const = 0;

private:
    Vertex *v_[2] = { nullptr, nullptr };
    RobustKernel *robust_ = nullptr;
    int param_id_ = -1;
};

template <int D, class E, class VertexXi, class VertexXj>
class BaseBinaryEdge : public Edge {
public:
    static const int Dimension = D;
    typedef E Measurement;
    typedef Matrix<double, D, D> InformationType;
    typedef Matrix<double, D, 1> ErrorVector;
    BaseBinaryEdge() : information_(InformationType::Identity()) {}
    const E &measurement() const { return measurement_; }
    void setMeasurement(const E &m) { measurement_ = m; }
    InformationType &information() { return information_; }
    const InformationType &information() const { return information_; }
    void setInformation(const InformationType &i) { information_ = i; }
    const ErrorVector &error() const { return error_; }   // filled by SparseOptimizer::computeActiveErrors
    double chi2() const override { return error_.dot(information_ * error_); }
    int dimension() const override { return D; }
    void packInformation(double *info) const override { for (int i = 0; i < D * D; ++i) info[i] = information_.data()[i]; }
    bool informationIsIdentity() const override { return information_.isIdentity(); }
    void unpackError(const double *e) override { for (int i = 0; i < D; ++i) error_[i] = e[i]; }

protected:
    E measurement_;
    InformationType information_;
    ErrorVector error_;
};

// ---- g2o::SE3Quat (row a17): x -> r x + t, tangent [omega, upsilon] ---------------------------------
class SE3Quat {
public:
    SE3Quat() {}
    SE3Quat(const Quaternion &q, const Vector3 &t) : r_(q), t_(t) { normalizeRotation(); }
    SE3Quat(const Matrix3 &R, const Vector3 &t) : r_(R), t_(t) { normalizeRotation(); }
    const Quaternion &rotation() const { return r_; }
    const Vector3 &translation() const { return t_; }
    void setRotation(const Quaternion &q) { r_ = q; }
    void setTranslation(const Vector3 &t) { t_ = t; }
    Vector3 map(const Vector3 &xyz) const { return r_ * xyz + t_; }
    SE3Quat inverse() const { const Quaternion ri = r_.conjugate(); return SE3Quat(ri, ri * (t_ * -1.0)); }
    SE3Quat operator*(const SE3Quat &o) const { return SE3Quat(r_ * o.r_, r_ * o.t_ + t_); }
    void normalizeRotation() {
        if (r_.w() < 0) r_ = Quaternion(-r_.w(), -r_.x(), -r_.y(), -r_.z());
        r_.normalize();
    }
    void pack(double *x) const { x[0] = r_.x(); x[1] = r_.y(); x[2] = r_.z(); x[3] = r_.w(); x[4] = t_[0]; x[5] = t_[1]; x[6] = t_[2]; }
    static SE3Quat unpack(const double *x) { SE3Quat T; T.r_ = Quaternion(x[3], x[0], x[1], x[2]); T.t_ = Vector3(x[4], x[5], x[6]); return T; }

private:
    Quaternion r_;
    Vector3 t_;
};

// ---- parameters (bal_example.cpp:90-96) -------------------------------------------------------------
class Parameter {
public:
    virtual ~Parameter() {}
    int id() const { return id_; }
    void setId(int id) { id_ = id; }

private:
    int id_ = -1;
};
class CameraParameters : public Parameter {
public:
    CameraParameters() : focal_length(1.0), baseline(0.5) {}
    CameraParameters(double f, const Matrix<double, 2, 1> &pp, double b) : focal_length(f), principle_point(pp), baseline(b) {}
    Matrix<double, 2, 1> cam_map(const Vector3 &x) const {
        Matrix<double, 2, 1> uv;
        uv[0] = x[0] / x[2] * focal_length + principle_point[0];
        uv[1] = x[1] / x[2] * focal_length + principle_point[1];
        return uv;
    }
    double focal_length;
    Matrix<double, 2, 1> principle_point;
    double baseline;
};

// ---- BA vertex / edge types (bal_example.cpp:113,:121,:143) ----------------------------------------
class VertexSE3Expmap : public BaseVertex<6, SE3Quat> {      // oplus: T <- exp(delta) T
public:
    int estimateDimension() const override { return 7; }
    int s3oKind() const override { return S3O_KIND_BA; }
    int baRole() const override { return 0; }
    void packEstimate(double *x) const override { estimate_.pack(x); }
    void unpackEstimate(const double *x) override { estimate_ = SE3Quat::unpack(x); }
};
class VertexSBAPointXYZ : public BaseVertex<3, Vector3> {     // oplus: p += delta
public:
    int estimateDimension() const override { return 3; }
    int s3oKind() const override { return S3O_KIND_BA; }
    int baRole() const override { return 1; }
    void packEstimate(double *x) const override { for (int i = 0; i < 3; ++i) x[i] = estimate_[i]; }
    void unpackEstimate(const double *x) override { for (int i = 0; i < 3; ++i) estimate_[i] = x[i]; }
};
// vertex(0) = point, vertex(1) = camera; e = z - cam_map(T.map(p))
class EdgeProjectXYZ2UV : public BaseBinaryEdge<2, Matrix<double, 2, 1>, VertexSBAPointXYZ, VertexSE3Expmap> {
public:
    int s3oKind() const override { return S3O_KIND_BA; }
    void packMeasurement(double *m) const override { m[0] = measurement_[0]; m[1] = measurement_[1]; }
    void computeError() {      // host-side read-out (bal_example.cpp:162-165); the solve evaluates on the device
        const VertexSE3Expmap *cam = static_cast<const VertexSE3Expmap *>(vertex(1));
        const VertexSBAPointXYZ *pt = static_cast<const VertexSBAPointXYZ *>(vertex(0));
        if (!cam || !pt || !camera_) return;
        error_ = measurement_ - camera_->cam_map(cam->estimate().map(pt->estimate()));
    }
    const CameraParameters *cameraParameters() const { return camera_; }

private:
    friend class SparseOptimizer;
    const CameraParameters *camera_ = nullptr;
};

// ---- solver plug-in slot (kitti_surf.cpp:553-557, :728-732; bal_example.cpp:73-83) --------------
template <class MatrixType>
class LinearSolver {
public:
    virtual ~LinearSolver() {}
    virtual bool init() { return true; }
};
// The reference's choice (SimplicialLDLT).  Here: a tag -- SparseOptimizer::optimize hands the whole LM to the device
// library, which picks its sparse block Cholesky or the multilevel PCG (s3o_set_linear_solver).  A LinearSolver that
// plugs into a REAL g2o block solver is in INTEGRATION.md (LinearSolverS3O over s3o_linsolver_solve).
template <class MatrixType>
class LinearSolverEigen : public LinearSolver<MatrixType> {};
template <class MatrixType>
class LinearSolverDense : public LinearSolver<MatrixType> {};

class Solver {
public:
    virtual ~Solver() {}
};
template <int PoseDim, int LandmarkDim>
class BlockSolver : public Solver {
public:
    struct PoseMatrixType {};
    struct LandmarkMatrixType {};
    typedef LinearSolver<PoseMatrixType> LinearSolverType;
    explicit BlockSolver(std::unique_ptr<LinearSolverType> linearSolver) : linear_(std::move(linearSolver)) {}
    LinearSolverType *linearSolver() const { return linear_.get(); }

private:
    std::unique_ptr<LinearSolverType> linear_;
};
typedef BlockSolver<-1, -1> BlockSolverX;
typedef BlockSolver<6, 3> BlockSolver_6_3;
typedef BlockSolver<7, 3> BlockSolver_7_3;

class OptimizationAlgorithm {
public:
    enum SolverResult { Terminate = 2, OK = 1, Fail = -1 };
    virtual ~OptimizationAlgorithm() {}
    virtual double tau() const { return 1e-5; }
    virtual double userLambdaInit() const { return 0; }
    virtual int maxTrialsAfterFailure() const { return 10; }
};
class OptimizationAlgorithmLevenberg : public OptimizationAlgorithm {
public:
    template <class SolverT>
    explicit OptimizationAlgorithmLevenberg(std::unique_ptr<SolverT> solver) : solver_(std::move(solver)) {}
    void setUserLambdaInit(double l) { user_lambda_ = l; }                 // kittiDetector.h:779-782
    void setMaxTrialsAfterFailure(int n) { max_trials_ = n; }              // kittiDetector.h:730
    double userLambdaInit() const override { return user_lambda_; }
    int maxTrialsAfterFailure() const override { return max_trials_; }
    double currentLambda() const { return current_lambda_; }
    int levenbergIteration() const { return lm_trials_; }

private:
    friend class SparseOptimizer;
    std::unique_ptr<Solver> solver_;
    double user_lambda_ = 0, current_lambda_ = 0;
    int max_trials_ = 10, lm_trials_ = 0;
};

// ---- g2o::SparseOptimizer ----------------------------------------------------------------------
class SparseOptimizer {
public:
    typedef std::map<int, Vertex *> VertexIDMap;
    typedef std::vector<Edge *> EdgeContainer;
    typedef std::vector<Vertex *> VertexContainer;

    SparseOptimizer() {}
    SparseOptimizer(const SparseOptimizer &) = delete;
    SparseOptimizer &operator=(const SparseOptimizer &) = delete;
    ~SparseOptimizer() {
        if (problem_) s3o_destroy(problem_);
        for (auto &kv : vertices_) delete kv.second;
        for (Edge *e : edges_) delete e;
        for (auto &kv : parameters_) delete kv.second;
        delete algorithm_;
    }
    bool addParameter(Parameter *prm) {                      // owned by the graph, as in g2o
        if (!prm || prm->id() < 0 || parameters_.count(prm->id())) return false;
        parameters_[prm->id()] = prm;
        return true;
    }
    Parameter *parameter(int id) const {
        auto it = parameters_.find(id);
        return it == parameters_.end() ? nullptr : it->second;
    }

    void setAlgorithm(OptimizationAlgorithm *a) { if (a != algorithm_) delete algorithm_; algorithm_ = a; }
    OptimizationAlgorithm *solver() const { return algorithm_; }
    OptimizationAlgorithm *algorithm() const { return algorithm_; }
    void setVerbose(bool v) { verbose_ = v; }
    bool verbose() const { return verbose_; }

    bool addVertex(Vertex *v) {
        if (!v || v->id() < 0 || vertices_.count(v->id())) return false;
        vertices_[v->id()] = v;
        initialized_ = false;
        return true;
    }
    bool addEdge(Edge *e) {
        if (!e || !e->vertex(0) || !e->vertex(1)) return false;
        for (int i = 0; i < 2; ++i) {
            auto it = vertices_.find(e->vertex(i)->id());
            if (it == vertices_.end() || it->second != e->vertex(i)) return false;
        }
        if (auto *proj = dynamic_cast<EdgeProjectXYZ2UV *>(e)) {   // g2o resolves parameters in addEdge
            proj->camera_ = dynamic_cast<const CameraParameters *>(parameter(e->parameterId()));
            if (!proj->camera_) return false;
        }
        edges_.push_back(e);
        initialized_ = false;
        return true;
    }
    Vertex *vertex(int id) const {
        auto it = vertices_.find(id);
        return it == vertices_.end() ? nullptr : it->second;
    }
    const VertexIDMap &vertices() const { return vertices_; }
    const EdgeContainer &edges() const { return edges_; }

    // device selection and B200-specific knobs (not part of g2o; all optional)
    void setDevice(int device) { device_ = device; }
    void setJacobianMode(int mode, double h = 1e-9) { jac_mode_ = mode; jac_h_ = h; }   // default: analytic
    void setMathMode(int mode) { math_mode_ = mode; }                                    // default: as written
    void setPcg(double rel_tol, int max_iter) { pcg_tol_ = rel_tol; pcg_max_iter_ = max_iter; }
    void setStopRelativeGain(double g) { stop_gain_ = g; }   // g2o's optional terminate action; 0 = off (reference)
    s3o_problem *problem() const { return problem_; }
    const std::string &lastError() const { return error_; }
    const std::vector<double> &history() const { return hist_; }   // per iteration [chi2, lambda, trials, rho, pcg]

    // SparseOptimizer::initializeOptimization [EXT g2o], call site kitti_surf.cpp:674: active
    // vertices sorted by id, edges in insertion order, Hessian indices assigned (fixed -> -1).
    bool initializeOptimization(int /*level*/ = 0) {
        initialized_ = false;
        if (vertices_.empty()) return fail("initializeOptimization: no vertices");
        const int kind = vertices_.begin()->second->s3oKind();
        for (auto &kv : vertices_)
            if (kv.second->s3oKind() != kind) return fail("initializeOptimization: mixed vertex kinds are not supported");
        for (Edge *e : edges_)
            if (e->s3oKind() != kind) return fail("initializeOptimization: edge kind does not match the vertices");
        if (problem_) { s3o_destroy(problem_); problem_ = nullptr; }
        if (s3o_create(kind, device_, &problem_) != S3O_OK) return fail(s3o_last_error());
        kind_ = kind;
        if (kind == S3O_KIND_BA) return initializeBA();
        const int n = (int)vertices_.size();
        const Vertex *first = vertices_.begin()->second;
        est_dim_ = first->estimateDimension();
        dim_ = first->dimension();
        order_.clear();
        dense_.clear();
        std::vector<uint8_t> fixed(n);
        std::vector<double> aux;
        for (auto &kv : vertices_) {           // std::map iterates in id order
            dense_[kv.first] = (int)order_.size();
            order_.push_back(kv.second);
        }
        est_.assign((size_t)n * est_dim_, 0.0);
        bool has_aux = false;
        double q4[4];
        for (int k = 0; k < n; ++k) {
            order_[k]->packEstimate(&est_[(size_t)k * est_dim_]);
            fixed[k] = order_[k]->fixed() ? 1 : 0;
            if (order_[k]->packAux(q4)) {
                if (!has_aux) { aux.assign((size_t)n * 4, 0.0); has_aux = true; }
                for (int c = 0; c < 4; ++c) aux[(size_t)k * 4 + c] = q4[c];
            }
        }
        if (s3o_set_vertices(problem_, n, est_.data(), fixed.data(), has_aux ? aux.data() : nullptr) != S3O_OK)
            return fail(s3o_last_error());
        const int ne = (int)edges_.size();
        std::vector<int32_t> v0(ne), v1(ne);
        std::vector<double> meas((size_t)ne * est_dim_), info;
        bool identity = true;
        for (Edge *e : edges_) identity = identity && e->informationIsIdentity();
        if (!identity) info.resize((size_t)ne * dim_ * dim_);
        const RobustKernel *rk = nullptr;
        for (int k = 0; k < ne; ++k) {
            Edge *e = edges_[k];
            v0[k] = dense_[e->vertex(0)->id()];
            v1[k] = dense_[e->vertex(1)->id()];
            e->packMeasurement(&meas[(size_t)k * est_dim_]);
            if (!identity) e->packInformation(&info[(size_t)k * dim_ * dim_]);
            if (!robustConsistent(e, k, rk)) return fail("initializeOptimization: the library applies ONE robust kernel to all edges; set the same kernel (kind and delta) on every edge or on none");
        }
        if (s3o_set_edges(problem_, ne, v0.data(), v1.data(), meas.data(), identity ? nullptr : info.data()) != S3O_OK)
            return fail(s3o_last_error());
        if (rk && s3o_set_robust(problem_, rk->s3oKind(), rk->delta()) != S3O_OK) return fail(s3o_last_error());
        s3o_set_jacobian_mode(problem_, jac_mode_, jac_h_);
        s3o_set_math_mode(problem_, math_mode_);
        if (pcg_tol_ > 0) s3o_set_pcg(problem_, pcg_tol_, pcg_max_iter_);
        int nf = 0, nb = 0;
        if (s3o_build_structure(problem_, &nf, &nb) != S3O_OK) return fail(s3o_last_error());
        std::vector<int32_t> hidx(n);
        if (s3o_get_hessian_index(problem_, hidx.data()) != S3O_OK) return fail(s3o_last_error());
        for (int k = 0; k < n; ++k) order_[k]->hessian_index_ = hidx[k];
        n_free_ = nf; n_blocks_ = nb;
        initialized_ = true;
        return true;
    }

    // SparseOptimizer::optimize [EXT g2o], call site kitti_surf.cpp:675.  Returns the number of
    // iterations performed, 0 when the first iteration fails, -1 when not initialised.
    int optimize(int iterations, bool /*online*/ = false) {
        if (!initialized_ || !problem_) { error_ = "optimize: initializeOptimization() has not succeeded"; return -1; }
        if (iterations <= 0) return 0;
        if (!uploadEstimates()) return -1;
        if (pcg_tol_ > 0) s3o_set_pcg(problem_, pcg_tol_, pcg_max_iter_);
        double tau = 1e-5, lam0 = 0;
        int max_trials = 10;
        if (algorithm_) { tau = algorithm_->tau(); lam0 = algorithm_->userLambdaInit(); max_trials = algorithm_->maxTrialsAfterFailure(); }
        s3o_set_lm(problem_, tau, lam0, max_trials);
        hist_.assign((size_t)iterations * 5, 0.0);
        int done = 0;
        double chi2 = 0, lambda = 0;
        if (s3o_optimize(problem_, iterations, stop_gain_, &done, &chi2, &lambda, hist_.data(), iterations) != S3O_OK) {
            error_ = s3o_last_error();
            return 0;
        }
        hist_.resize((size_t)std::max(done, 0) * 5);
        if (auto *lm = dynamic_cast<OptimizationAlgorithmLevenberg *>(algorithm_)) {
            lm->current_lambda_ = lambda;
            lm->lm_trials_ = done > 0 ? (int)hist_[(size_t)(done - 1) * 5 + 2] : 0;
        }
        if (verbose_)
            for (int it = 0; it < done; ++it)
                std::fprintf(stderr, "iteration= %d\t chi2= %.6f\t edges= %d\t schur= 0\t lambda= %.6f\t levenbergIter= %d\t pcgIter= %d\n",
                             it, hist_[(size_t)it * 5], (int)edges_.size(), hist_[(size_t)it * 5 + 1],
                             (int)hist_[(size_t)it * 5 + 2], (int)hist_[(size_t)it * 5 + 4]);
        if (!downloadEstimates()) return 0;
        chi2_ = chi2;
        return done;
    }

    // computeActiveErrors + activeChi2 / activeRobustChi2 (kittiDetector.h:928-950 style read-outs)
    void computeActiveErrors() {
        if (!initialized_ || !uploadEstimates()) return;
        const int ed = kind_ == S3O_KIND_BA ? 2 : dim_;
        std::vector<double> err((size_t)edges_.size() * ed);
        if (s3o_edge_errors(problem_, err.data()) != S3O_OK) { error_ = s3o_last_error(); return; }
        if (kind_ == S3O_KIND_BA) {
            for (size_t k = 0; k < edges_.size(); ++k) edges_[k]->unpackError(&err[k * 2]);
            if (s3o_chi2(problem_, &chi2_) != S3O_OK) error_ = s3o_last_error();
            return;
        }
        for (size_t k = 0; k < edges_.size(); ++k) edges_[k]->unpackError(&err[k * dim_]);
        if (s3o_chi2(problem_, &chi2_) != S3O_OK) error_ = s3o_last_error();
    }
    // SparseOptimizer::computeMarginals [EXT g2o]: blocks (hessianIndex, hessianIndex) of H^-1 at the vertices' current
    // estimates (s3o_compute_marginals; for BA s3o_ba_compute_marginals, where a block row / column is 6 wide for a
    // camera and 3 for a point).  spinv gets one block row / column per free vertex and the requested blocks.  A vertex
    // without a Hessian index (fixed) makes the call fail.
    bool computeMarginals(SparseBlockMatrix<MatrixX> &spinv, const std::vector<std::pair<int, int>> &blockIndices) {
        if (!initialized_ || !problem_) return fail("computeMarginals: initializeOptimization() has not succeeded");
        if (!uploadEstimates()) return false;
        const bool ba = kind_ == S3O_KIND_BA;
        const int nb = ba ? n_free_ + n_free_points_ : n_free_;
        auto dim = [&](int h) { return ba && h >= n_free_ ? 3 : dim_; };
        const int m = (int)blockIndices.size();
        std::vector<int32_t> rows(m), cols(m);
        std::vector<size_t> off(m + 1, 0);
        for (int k = 0; k < m; ++k) {
            rows[k] = blockIndices[k].first; cols[k] = blockIndices[k].second;
            off[k + 1] = off[k] + (size_t)dim(rows[k]) * dim(cols[k]);
        }
        std::vector<double> out(off[m]);
        if (m > 0 && (ba ? s3o_ba_compute_marginals(problem_, m, rows.data(), cols.data(), out.data())
                         : s3o_compute_marginals(problem_, m, rows.data(), cols.data(), out.data())) != S3O_OK)
            return fail(s3o_last_error());
        std::vector<int> bi(nb);
        for (int k = 0; k < nb; ++k) bi[k] = (k ? bi[k - 1] : 0) + dim(k);
        spinv = SparseBlockMatrix<MatrixX>(bi.data(), bi.data(), nb, nb);
        for (int k = 0; k < m; ++k) {
            MatrixX *b = spinv.block(rows[k], cols[k], true);
            std::copy(out.begin() + off[k], out.begin() + off[k + 1], b->data());
        }
        return true;
    }
    bool computeMarginals(SparseBlockMatrix<MatrixX> &spinv, const Vertex *vertex) {
        if (!vertex || vertex->hessianIndex() < 0) return false;
        return computeMarginals(spinv, std::vector<std::pair<int, int>>{ { vertex->hessianIndex(), vertex->hessianIndex() } });
    }
    bool computeMarginals(SparseBlockMatrix<MatrixX> &spinv, const VertexContainer &vertices) {
        std::vector<std::pair<int, int>> indices;
        for (const Vertex *v : vertices) indices.push_back({ v->hessianIndex(), v->hessianIndex() });
        return computeMarginals(spinv, indices);
    }

    double activeChi2() const { double s = 0; for (Edge *e : edges_) s += e->chi2(); return s; }
    double activeRobustChi2() const { return chi2_; }
    int numFreeVertices() const { return n_free_; }
    int numHessianBlocks() const { return n_blocks_; }
    // g2o-order upper block-CCS of Hpp (BlockSolver::buildStructure), for structure checks
    bool hessianStructure(std::vector<int32_t> &colptr, std::vector<int32_t> &rowidx) const {
        if (!initialized_) return false;
        colptr.resize(n_free_ + 1);
        rowidx.resize(n_blocks_);
        return s3o_get_structure(problem_, colptr.data(), rowidx.data()) == S3O_OK;
    }

private:
    // s3o_set_robust is per problem: every edge must carry the same kernel (kind, delta) or none (edge k of the scan)
    static bool robustConsistent(const Edge *e, int k, const RobustKernel *&rk) {
        const RobustKernel *r = e->robustKernel();
        if (k == 0) { rk = r; return true; }
        if ((r == nullptr) != (rk == nullptr)) return false;
        return !r || (r->s3oKind() == rk->s3oKind() && r->delta() == rk->delta());
    }
    bool fail(const char *msg) { error_ = msg ? msg : "unknown error"; return false; }
    // BA graph (bal_example.cpp:98-198): cameras and points in id order, observations in insertion order
    bool initializeBA() {
        order_.clear(); points_.clear(); dense_.clear();
        for (auto &kv : vertices_) {
            Vertex *v = kv.second;
            if (v->baRole() == 0) { dense_[kv.first] = (int)order_.size(); order_.push_back(v); }
            else if (v->baRole() == 1) { dense_[kv.first] = (int)points_.size(); points_.push_back(v); }
            else return fail("initializeOptimization: unknown vertex type in a BA graph");
        }
        const int nc = (int)order_.size(), np = (int)points_.size(), ne = (int)edges_.size();
        est_.assign((size_t)nc * 7, 0.0);
        pts_.assign((size_t)np * 3, 0.0);
        std::vector<uint8_t> cfix(nc), pfix(np);
        for (int k = 0; k < nc; ++k) { order_[k]->packEstimate(&est_[(size_t)k * 7]); cfix[k] = order_[k]->fixed(); }
        for (int k = 0; k < np; ++k) { points_[k]->packEstimate(&pts_[(size_t)k * 3]); pfix[k] = points_[k]->fixed(); }
        std::vector<int32_t> oc(ne), op(ne);
        std::vector<double> uv((size_t)ne * 2), info;
        bool identity = true;
        for (Edge *e : edges_) identity = identity && e->informationIsIdentity();
        if (!identity) info.resize((size_t)ne * 3);
        const RobustKernel *rk = nullptr;
        const CameraParameters *cam = nullptr;
        for (int k = 0; k < ne; ++k) {
            Edge *e = edges_[k];
            if (e->vertex(0)->baRole() != 1 || e->vertex(1)->baRole() != 0) return fail("initializeOptimization: EdgeProjectXYZ2UV needs vertex(0) = point, vertex(1) = camera");
            op[k] = dense_[e->vertex(0)->id()];
            oc[k] = dense_[e->vertex(1)->id()];
            e->packMeasurement(&uv[(size_t)k * 2]);
            if (!identity) { double m[4]; e->packInformation(m); info[(size_t)k * 3] = m[0]; info[(size_t)k * 3 + 1] = m[1]; info[(size_t)k * 3 + 2] = m[3]; }
            if (!robustConsistent(e, k, rk)) return fail("initializeOptimization: the library applies ONE robust kernel to all edges; set the same kernel (kind and delta) on every edge or on none");
            if (auto *proj = dynamic_cast<EdgeProjectXYZ2UV *>(e)) cam = proj->cameraParameters();
        }
        if (!cam) return fail("initializeOptimization: no CameraParameters (addParameter + setParameterId)");
        if (s3o_ba_set_cameras(problem_, nc, est_.data(), cfix.data()) != S3O_OK ||
            s3o_ba_set_points(problem_, np, pts_.data(), pfix.data()) != S3O_OK ||
            s3o_ba_set_observations(problem_, ne, oc.data(), op.data(), uv.data(), identity ? nullptr : info.data()) != S3O_OK ||
            s3o_ba_set_intrinsics(problem_, cam->focal_length, cam->principle_point[0], cam->principle_point[1]) != S3O_OK)
            return fail(s3o_last_error());
        if (rk && s3o_set_robust(problem_, rk->s3oKind(), rk->delta()) != S3O_OK) return fail(s3o_last_error());
        if (pcg_tol_ > 0) s3o_set_pcg(problem_, pcg_tol_, pcg_max_iter_);
        int nf = 0, nb = 0;
        if (s3o_build_structure(problem_, &nf, &nb) != S3O_OK) return fail(s3o_last_error());
        int hc = 0, hp = 0;      // free cameras numbered first, then the marginalised points
        for (Vertex *v : order_) v->hessian_index_ = v->fixed() ? -1 : hc++;
        for (Vertex *v : points_) v->hessian_index_ = v->fixed() ? -1 : hc + hp++;
        est_dim_ = 7; dim_ = 6; n_free_ = nf; n_free_points_ = hp; n_blocks_ = nb;
        initialized_ = true;
        return true;
    }
    bool uploadEstimates() {
        if (kind_ == S3O_KIND_BA) {
            for (size_t k = 0; k < order_.size(); ++k) order_[k]->packEstimate(&est_[k * 7]);
            for (size_t k = 0; k < points_.size(); ++k) points_[k]->packEstimate(&pts_[k * 3]);
            if (s3o_ba_set_estimates(problem_, est_.data(), pts_.data()) != S3O_OK) { error_ = s3o_last_error(); return false; }
            return true;
        }
        for (size_t k = 0; k < order_.size(); ++k) order_[k]->packEstimate(&est_[k * est_dim_]);
        if (s3o_set_estimates(problem_, est_.data()) != S3O_OK) { error_ = s3o_last_error(); return false; }
        return true;
    }
    bool downloadEstimates() {
        if (kind_ == S3O_KIND_BA) {
            if (s3o_ba_get_cameras(problem_, est_.data()) != S3O_OK || s3o_ba_get_points(problem_, pts_.data()) != S3O_OK) { error_ = s3o_last_error(); return false; }
            for (size_t k = 0; k < order_.size(); ++k) if (!order_[k]->fixed()) order_[k]->unpackEstimate(&est_[k * 7]);
            for (size_t k = 0; k < points_.size(); ++k) if (!points_[k]->fixed()) points_[k]->unpackEstimate(&pts_[k * 3]);
            return true;
        }
        if (s3o_get_vertices(problem_, est_.data()) != S3O_OK) { error_ = s3o_last_error(); return false; }
        for (size_t k = 0; k < order_.size(); ++k)
            if (!order_[k]->fixed()) order_[k]->unpackEstimate(&est_[k * est_dim_]);
        return true;
    }

    VertexIDMap vertices_;
    EdgeContainer edges_;
    OptimizationAlgorithm *algorithm_ = nullptr;
    s3o_problem *problem_ = nullptr;
    std::vector<Vertex *> order_, points_;      // pose-graph vertices or BA cameras; BA points
    std::map<int, int> dense_;
    std::map<int, Parameter *> parameters_;
    std::vector<double> est_, pts_, hist_;
    std::string error_;
    bool verbose_ = false, initialized_ = false;
    int device_ = 0, kind_ = 0, est_dim_ = 0, dim_ = 0, n_free_ = 0, n_free_points_ = 0, n_blocks_ = 0;
    int jac_mode_ = S3O_JAC_ANALYTIC, math_mode_ = S3O_MATH_REFERENCE, pcg_max_iter_ = 0;
    double jac_h_ = 1e-9, pcg_tol_ = 0, stop_gain_ = 0, chi2_ = 0;
};

}  // namespace g2o

// ---- vio_g2o types used by the reference (rows a9, a10, a18) ------------------------------------
namespace vio {

// Fixed rotation carried by a scale+translation vertex (the reference stores a Sophus::SO3d,
// kitti_surf.cpp:792-793, and reads it back with unit_quaternion(), :1035).
class SO3 {
public:
    SO3() {}
    explicit SO3(const g2o::Matrix3 &R) : q_(R) {}
    explicit SO3(const g2o::Quaternion &q) : q_(q) {}
    const g2o::Quaternion &unit_quaternion() const { return q_; }
    g2o::Matrix3 matrix() const { return q_.toRotationMatrix(); }

private:
    g2o::Quaternion q_;
};

class VertexSim3Expmap : public g2o::BaseVertex<7, g2o::Sim3> {   // oplus: S <- exp(delta) S
public:
    int estimateDimension() const override { return 8; }
    int s3oKind() const override { return S3O_KIND_SIM3; }
    void packEstimate(double *x) const override { estimate_.pack(x); }
    void unpackEstimate(const double *x) override { estimate_ = g2o::Sim3::unpack(x); }
};
class EdgeSim3 : public g2o::BaseBinaryEdge<7, g2o::Sim3, VertexSim3Expmap, VertexSim3Expmap> {
public:   // e = log(C * S_v0 * S_v1^-1)
    int s3oKind() const override { return S3O_KIND_SIM3; }
    void packMeasurement(double *m) const override { measurement_.pack(m); }
};

class G2oVertexScale : public g2o::BaseVertex<1, double> {
public:
    G2oVertexScale() { estimate_ = 1.0; }
    int estimateDimension() const override { return 1; }
    int s3oKind() const override { return S3O_KIND_SCALE; }
    void packEstimate(double *x) const override { x[0] = estimate_; }
    void unpackEstimate(const double *x) override { estimate_ = x[0]; }
};
class G2oEdgeScale : public g2o::BaseBinaryEdge<1, double, G2oVertexScale, G2oVertexScale> {
public:
    G2oEdgeScale() { measurement_ = 1.0; }
    int s3oKind() const override { return S3O_KIND_SCALE; }
    void packMeasurement(double *m) const override { m[0] = measurement_; }
};

class G2oVertexScaleTrans : public g2o::BaseVertex<4, g2o::Vector4> {   // [s_w2i, t_w2i]
public:
    SO3 Rw2i;
    int estimateDimension() const override { return 4; }
    int s3oKind() const override { return S3O_KIND_SCALE_TRANS; }
    void packEstimate(double *x) const override { for (int i = 0; i < 4; ++i) x[i] = estimate_[i]; }
    void unpackEstimate(const double *x) override { for (int i = 0; i < 4; ++i) estimate_[i] = x[i]; }
    bool packAux(double *q) const override {
        const g2o::Quaternion &u = Rw2i.unit_quaternion();
        q[0] = u.x(); q[1] = u.y(); q[2] = u.z(); q[3] = u.w();
        return true;
    }
};
class G2oEdgeScaleTrans : public g2o::BaseBinaryEdge<4, g2o::Vector4, G2oVertexScaleTrans, G2oVertexScaleTrans> {
public:
    int s3oKind() const override { return S3O_KIND_SCALE_TRANS; }
    void packMeasurement(double *m) const override { for (int i = 0; i < 4; ++i) m[i] = measurement_[i]; }
};

}  // namespace vio
