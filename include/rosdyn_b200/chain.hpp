// chain.hpp -- C++ facade over the C-ABI (rosdyn_b200.h) with the method names of rosdyn::Chain
// (reference: rosdyn_core/include/rosdyn_core/primitives.h:235-555).
//
// * per-sample getters take/return std containers laid out exactly like the reference's Eigen objects
//   (column-major matrices, 6-vectors linear-then-angular) and run as N = 1 batches on the GPU;
// * batched siblings take SoA arrays (host or device) and forward to the C-ABI;
// * Eigen-typed overloads with the reference's signatures appear when <Eigen/Core> is available.  Eigen3 is not in the build image; they are
//   compile-tested against the Eigen subset of oracle/shim (tests/test_cpp_headers.py) and use element access only.
// Errors follow the reference: std::runtime_error from the constructor (primitives_impl.h:498-501),
// std::invalid_argument("Input data dimensions mismatch") from getRegressor (primitives_impl.h:1299-1309).
// Like the reference class, one object serves one thread at a time.
#ifndef ROSDYN_B200_CHAIN_HPP
#define ROSDYN_B200_CHAIN_HPP

#include <array>
#include <cmath>
#include <stdexcept>
#include <string>
#include <vector>

#include "../rosdyn_b200.h"

#if defined(__has_include)
#if __has_include(<Eigen/Core>)
#include <Eigen/Core>
#include <Eigen/Geometry>
#include <Eigen/StdVector>
#define ROSDYN_B200_HAVE_EIGEN 1
#endif
#endif

namespace rosdyn_b200
{

using Vector6d = std::array<double, 6>;
using VectorXd = std::vector<double>;
using Affine3dImage = std::array<double, 16>;  // 4x4 column-major, the memory image of Eigen::Affine3d

// URDF rpy -> row-major rotation, R = Rz(yaw) Ry(pitch) Rx(roll) (urdf_parser.h:44-50 via the URDF quaternion)
inline void rpyToRot(double r, double p, double y, double R[9])
{
  const double cr = std::cos(r), sr = std::sin(r), cp = std::cos(p), sp = std::sin(p), cy = std::cos(y), sy = std::sin(y);
  R[0] = cy * cp; R[1] = cy * sp * sr - sy * cr; R[2] = cy * sp * cr + sy * sr;
  R[3] = sy * cp; R[4] = sy * sp * sr + cy * cr; R[5] = sy * sp * cr - cy * sr;
  R[6] = -sp;     R[7] = cp * sr;                R[8] = cp * cr;
}

class Chain
{
public:
  explicit Chain(const rdb_chain_desc& desc)
  {
    const rdb_status s = rdb_chain_create(&desc, &m_h);
    if (s != RDB_OK) throw std::runtime_error(std::string("rosdyn_b200: ") + rdb_last_error());
    m_nj = rdb_chain_joints_number(m_h);
    m_nl = rdb_chain_links_number(m_h);
    m_n = rdb_chain_active_joints_number(m_h);
  }
  // Chain(robot_description, base_link_name, ee_link_name, gravity) (primitives.h:349-352); throws std::runtime_error
  // ("Base link not found" / "Tool link not found", primitives_impl.h:498-501) like the reference
  Chain(const std::string& robot_description, const std::string& base_link_name, const std::string& ee_link_name,
        const std::array<double, 3>& gravity = {0.0, 0.0, 0.0})
  {
    const rdb_status s = rdb_chain_from_urdf(robot_description.c_str(), base_link_name.c_str(), ee_link_name.c_str(), gravity.data(), &m_h);
    if (s != RDB_OK) throw std::runtime_error(rdb_last_error());
    m_nj = rdb_chain_joints_number(m_h);
    m_nl = rdb_chain_links_number(m_h);
    m_n = rdb_chain_active_joints_number(m_h);
  }
  ~Chain() { rdb_chain_destroy(m_h); }
  Chain(const Chain&) = delete;
  Chain& operator=(const Chain&) = delete;

  unsigned int getLinksNumber() const { return m_nl; }
  unsigned int getJointsNumber() const { return m_nj; }
  unsigned int getActiveJointsNumber() const { return m_n; }
  const rdb_chain* handle() const { return m_h; }
  rdb_chain* handle() { return m_h; }
  std::array<double, 3> getGravity() const
  {
    std::array<double, 3> g{};
    rdb_chain_gravity(m_h, g.data());
    return g;
  }
  VectorXd getNominalParameters() const
  {
    VectorXd p(10 * m_nj);
    rdb_chain_nominal_parameters(m_h, p.data());
    return p;
  }
  // Chain::setInputJointsName by chain-joint index (primitives_impl.h:705-742)
  bool setInputJoints(const std::vector<int32_t>& chain_joint_of_input)
  {
    check(rdb_chain_set_input_joints(m_h, (int32_t)chain_joint_of_input.size(), chain_joint_of_input.data()));
    m_n = rdb_chain_active_joints_number(m_h);
    for (int32_t j : chain_joint_of_input)
      if (j < 0 || j >= (int32_t)m_nj) return false;
    return true;
  }

  // ---------------------------------------------------------------- per-sample getters (reference names)
  // poses come back in the Eigen-record layout of the ABI (RDB_LAYOUT_EIGEN): 16 doubles = the memory image of Eigen::Affine3d
  Affine3dImage getTransformation(const VectorXd& q)
  {
    const VectorXd t = kin1(q, nullptr, nullptr, nullptr, &rdb_kinematics_out::T_tool, 16, RDB_LAYOUT_EIGEN);
    Affine3dImage T{};
    for (int k = 0; k < 16; k++) T[k] = t[k];
    return T;
  }
  std::vector<Affine3dImage> getTransformations(const VectorXd& q)
  {
    const VectorXd t = kin1(q, nullptr, nullptr, nullptr, &rdb_kinematics_out::T_links, 16 * m_nl, RDB_LAYOUT_EIGEN);
    std::vector<Affine3dImage> out(m_nl);
    for (unsigned l = 0; l < m_nl; l++)
      for (int k = 0; k < 16; k++) out[l][k] = t[16 * l + k];
    return out;
  }
  // 6 x n_act, column-major
  VectorXd getJacobian(const VectorXd& q) { return kin1(q, nullptr, nullptr, nullptr, &rdb_kinematics_out::jacobian, 6 * m_n); }
  std::vector<Vector6d> getTwist(const VectorXd& q, const VectorXd& Dq) { return six(kin1(q, &Dq, nullptr, nullptr, &rdb_kinematics_out::twist, 6 * m_nl)); }
  Vector6d getTwistTool(const VectorXd& q, const VectorXd& Dq) { return getTwist(q, Dq).back(); }
  std::vector<Vector6d> getDTwist(const VectorXd& q, const VectorXd& Dq, const VectorXd& DDq)
  {
    return six(kin1(q, &Dq, &DDq, nullptr, &rdb_kinematics_out::dtwist, 6 * m_nl));
  }
  Vector6d getDTwistTool(const VectorXd& q, const VectorXd& Dq, const VectorXd& DDq) { return getDTwist(q, Dq, DDq).back(); }
  std::vector<Vector6d> getDTwistLinearPart(const VectorXd& q, const VectorXd& DDq)
  {
    return six(kin1(q, nullptr, &DDq, nullptr, &rdb_kinematics_out::dtwist_lin, 6 * m_nl));
  }
  std::vector<Vector6d> getDTwistNonLinearPart(const VectorXd& q, const VectorXd& Dq)
  {
    return six(kin1(q, &Dq, nullptr, nullptr, &rdb_kinematics_out::dtwist_nonlin, 6 * m_nl));
  }
  std::vector<Vector6d> getDDTwist(const VectorXd& q, const VectorXd& Dq, const VectorXd& DDq, const VectorXd& DDDq)
  {
    return six(kin1(q, &Dq, &DDq, &DDDq, &rdb_kinematics_out::ddtwist, 6 * m_nl));
  }
  Vector6d getDDTwistTool(const VectorXd& q, const VectorXd& Dq, const VectorXd& DDq, const VectorXd& DDDq)
  {
    return getDDTwist(q, Dq, DDq, DDDq).back();
  }
  std::vector<Vector6d> getDDTwistLinearPart(const VectorXd& q, const VectorXd& DDDq)
  {
    return six(kin1(q, nullptr, nullptr, &DDDq, &rdb_kinematics_out::ddtwist_lin, 6 * m_nl));
  }
  std::vector<Vector6d> getDDTwistNonLinearPart(const VectorXd& q, const VectorXd& Dq, const VectorXd& DDq)
  {
    return six(kin1(q, &Dq, &DDq, nullptr, &rdb_kinematics_out::ddtwist_nonlin, 6 * m_nl));
  }
  VectorXd getJointTorque(const VectorXd& q, const VectorXd& Dq, const VectorXd& DDq)
  {
    sizes(q, &Dq, &DDq, nullptr);
    VectorXd tau(m_n);
    rdb_samples in{1, 1, q.data(), Dq.data(), DDq.data(), nullptr};
    check(rdb_torque_batch_host(m_h, &in, tau.data(), 1));
    return tau;
  }
  VectorXd getJointTorqueNonLinearPart(const VectorXd& q, const VectorXd& Dq)
  {
    sizes(q, &Dq, nullptr, nullptr);
    VectorXd tau(m_n);
    rdb_samples in{1, 1, q.data(), Dq.data(), nullptr, nullptr};
    check(rdb_torque_batch_host(m_h, &in, tau.data(), 1));
    return tau;
  }
  // forward dynamics ddq = M(q)^-1 (tau - h(q, Dq)) (rdb_forward_dynamics_batch); all NaN when M(q) is not positive definite
  VectorXd getJointAcceleration(const VectorXd& q, const VectorXd& Dq, const VectorXd& tau)
  {
    sizes(q, &Dq, &tau, nullptr);
    VectorXd ddq(m_n);
    rdb_samples in{1, 1, q.data(), Dq.data(), nullptr, nullptr};
    check(rdb_forward_dynamics_batch_host(m_h, &in, tau.data(), ddq.data(), 1, nullptr));
    return ddq;
  }
  // n_act x 10 nJ, column-major (the memory image of the Eigen::MatrixXd the reference returns by value)
  VectorXd getRegressor(const VectorXd& q, const VectorXd& Dq, const VectorXd& DDq)
  {
    if (q.size() != Dq.size() || Dq.size() != DDq.size() || q.size() != m_n) throw std::invalid_argument("Input data dimensions mismatch");
    VectorXd phi((size_t)10 * m_nj * m_n);
    rdb_samples in{1, 1, q.data(), Dq.data(), DDq.data(), nullptr};
    check(rdb_regressor_batch_host(m_h, &in, phi.data(), nullptr, 1));
    return phi;
  }
  // n_act x n_act, column-major
  VectorXd getJointInertia(const VectorXd& q)
  {
    sizes(q, nullptr, nullptr, nullptr);
    VectorXd M((size_t)m_n * m_n);
    rdb_samples in{1, 1, q.data(), nullptr, nullptr, nullptr};
    check(rdb_inertia_batch_host(m_h, &in, M.data(), 1));
    return M;
  }

  // ---------------------------------------------------------------- batched siblings (SoA planes, see rosdyn_b200.h)
  // device pointers, asynchronous on `stream` (a cudaStream_t)
  void computeTransformations(const rdb_samples& in, const rdb_kinematics_out& out, void* stream = nullptr) { check(rdb_kinematics_batch(m_h, &in, &out, stream)); }
  void getJointTorque(const rdb_samples& in, double* torque, int64_t ld_out, void* stream = nullptr) { check(rdb_torque_batch(m_h, &in, torque, ld_out, stream)); }
  void getRegressor(const rdb_samples& in, double* phi, double* torque, int64_t ld_out, void* stream = nullptr)
  {
    check(rdb_regressor_batch(m_h, &in, phi, torque, ld_out, stream));
  }
  void getJointInertia(const rdb_samples& in, double* inertia, int64_t ld_out, void* stream = nullptr) { check(rdb_inertia_batch(m_h, &in, inertia, ld_out, stream)); }
  // tau [n_act][in.ld] (nullptr = 0), ddq [n_act][ld_out], info [n] optional (1 = M not positive definite)
  void getJointAcceleration(const rdb_samples& in, const double* tau, double* ddq, int64_t ld_out, int32_t* info = nullptr, void* stream = nullptr)
  {
    check(rdb_forward_dynamics_batch(m_h, &in, tau, ddq, ld_out, info, stream));
  }
  void getRegressorGram(const rdb_samples& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq, bool accumulate, void* stream = nullptr)
  {
    check(rdb_regressor_gram_batch(m_h, &in, tau_meas, gram, rhs, tau_sq, accumulate ? 1 : 0, stream));
  }
  // Chain::getWrench / getJointTorque(q,Dq,DDq,ext_wrenches_in_link_frame) (primitives_impl.h:1225-1274); ext [nL][6][ld_ext] or nullptr
  void getWrench(const rdb_samples& in, const double* ext_wrenches, int64_t ld_ext, double* torque, double* wrenches, int64_t ld_out, void* stream = nullptr)
  {
    check(rdb_wrench_batch(m_h, &in, ext_wrenches, ld_ext, torque, wrenches, ld_out, stream));
  }
  // Chain::getJacobianLink (primitives_impl.h:951-979) by link index; std::invalid_argument for a link outside the chain (:960)
  void getJacobianLink(const rdb_samples& in, int32_t link_index, double* jacobian, int64_t ld_out, void* stream = nullptr)
  {
    const rdb_status s = rdb_jacobian_link_batch(m_h, &in, link_index, jacobian, ld_out, stream);
    if (s == RDB_ERR_NOT_FOUND) throw std::invalid_argument(rdb_last_error());
    check(s);
  }
  // Chain::computeLocalIk / computeWeigthedLocalIk (primitives_impl.h:1398-1468) for n target poses (device planes: target[12][ld] 3x4
  // row-major, seed / sol [n_act][ld]); the wall-clock budget of the reference is an iteration budget.  q_min / q_max / weight: host
  // arrays or nullptr (no limits / unweighted).  status[i] = 1 where the reference would return true.
  void computeLocalIk(int64_t n, int64_t ld, const double* target, const double* seed, const double* q_min, const double* q_max,
                      const double* weight, double toll, int32_t max_iter, double* sol, int32_t* status = nullptr,
                      int32_t* iterations = nullptr, double* error_norm = nullptr, void* stream = nullptr)
  {
    check(rdb_local_ik_batch(m_h, n, ld, target, seed, q_min, q_max, weight, toll, max_iter, sol, status, iterations, error_norm, stream));
  }
  // one process, several GPUs: contiguous shards of a HOST batch on the given chains (one per device, see rdb_chain_create_on), partial
  // normal equations summed on the host in rank order
  static void regressorGramSharded(const std::vector<Chain*>& chains, const rdb_samples& in, const double* tau_meas, double* gram, double* rhs,
                                   double* tau_sq, bool accumulate = false)
  {
    std::vector<rdb_chain*> h;
    for (Chain* c : chains) h.push_back(c->m_h);
    check(rdb_regressor_gram_sharded_host(h.data(), (int32_t)h.size(), &in, tau_meas, gram, rhs, tau_sq, accumulate ? 1 : 0));
  }
  // Chain::getMultiplicity (primitives_impl.h:1470-1517): multi-turn images of q inside [q_min, q_max]; joint_type_of_input[i] = RDB_JOINT_*
  static std::vector<std::vector<double>> getMultiplicity(const std::vector<int32_t>& joint_type_of_input, const std::vector<double>& q,
                                                          const std::vector<double>& q_min, const std::vector<double>& q_max)
  {
    const int32_t n = (int32_t)q.size();
    int64_t count = 0;
    rdb_multiplicity(n, joint_type_of_input.data(), q.data(), q_min.data(), q_max.data(), nullptr, 0, &count);
    std::vector<double> flat((size_t)count * n);
    check(rdb_multiplicity(n, joint_type_of_input.data(), q.data(), q_min.data(), q_max.data(), flat.data(), count, &count));
    std::vector<std::vector<double>> out((size_t)count);
    for (int64_t k = 0; k < count; k++) out[k].assign(flat.begin() + k * n, flat.begin() + (k + 1) * n);
    return out;
  }
  // additive joint components (friction_polynomial1.h, friction_polynomial2.h, ideal_spring.h) as extra regressor columns
  unsigned int setComponents(const std::vector<rdb_component_desc>& components)
  {
    const rdb_status s = rdb_chain_set_components(m_h, (int32_t)components.size(), components.data());
    if (s == RDB_ERR_NOT_FOUND) throw std::invalid_argument(rdb_last_error());  // ComponentBase ctor, base_component.h:103-104
    check(s);
    return (unsigned int)rdb_chain_component_columns(m_h);
  }
  unsigned int getComponentColumns() const { return (unsigned int)rdb_chain_component_columns(m_h); }
  void getComponentsRegressor(const rdb_samples& in, double* phi_c, int64_t ld_out, void* stream = nullptr)
  {
    check(rdb_components_regressor_batch(m_h, &in, phi_c, ld_out, stream));
  }
  void getComponentsTorque(const rdb_samples& in, const VectorXd& parameters, double* torque, int64_t ld_out, bool accumulate, void* stream = nullptr)
  {
    if (parameters.size() != getComponentColumns()) throw std::invalid_argument("Input data dimensions mismatch");
    check(rdb_components_torque_batch(m_h, &in, parameters.data(), torque, ld_out, accumulate ? 1 : 0, stream));
  }
  void getRegressorGramExt(const rdb_samples& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq, bool accumulate, void* stream = nullptr)
  {
    check(rdb_regressor_gram_ext_batch(m_h, &in, tau_meas, gram, rhs, tau_sq, accumulate ? 1 : 0, stream));
  }
  // minimum-norm solution of the normal equations (host arrays); returns the rank
  static int solveNormalEquations(const VectorXd& gram, const VectorXd& rhs, double tau_sq, VectorXd& parameters, double* residual_sq = nullptr,
                                  double rel_tol = 1e-10)
  {
    const int32_t P = (int32_t)rhs.size();
    if (gram.size() != (size_t)P * P) throw std::invalid_argument("Input data dimensions mismatch");
    parameters.assign(P, 0.0);
    int32_t rank = 0;
    check(rdb_normal_equations_solve(P, gram.data(), rhs.data(), tau_sq, rel_tol, parameters.data(), nullptr, &rank, residual_sq));
    return rank;
  }
  // host pointers (copies and synchronisation inside)
  void computeTransformationsHost(const rdb_samples& in, const rdb_kinematics_out& out) { check(rdb_kinematics_batch_host(m_h, &in, &out)); }
  void getJointTorqueHost(const rdb_samples& in, double* torque, int64_t ld_out) { check(rdb_torque_batch_host(m_h, &in, torque, ld_out)); }
  void getRegressorHost(const rdb_samples& in, double* phi, double* torque, int64_t ld_out) { check(rdb_regressor_batch_host(m_h, &in, phi, torque, ld_out)); }
  void getJointInertiaHost(const rdb_samples& in, double* inertia, int64_t ld_out) { check(rdb_inertia_batch_host(m_h, &in, inertia, ld_out)); }
  void getJointAccelerationHost(const rdb_samples& in, const double* tau, double* ddq, int64_t ld_out, int32_t* info = nullptr)
  {
    check(rdb_forward_dynamics_batch_host(m_h, &in, tau, ddq, ld_out, info));
  }
  void getRegressorGramHost(const rdb_samples& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq, bool accumulate)
  {
    check(rdb_regressor_gram_batch_host(m_h, &in, tau_meas, gram, rhs, tau_sq, accumulate ? 1 : 0));
  }

#ifdef ROSDYN_B200_HAVE_EIGEN
  // ---------------------------------------------------------------- Eigen-typed drop-ins: the reference's signatures (primitives.h:452-548).
  // Results are returned BY VALUE (the reference returns const& to member caches that the next call overwrites).  Written with element access
  // only, so that they compile with Eigen3 proper and with the Eigen subset of oracle/shim (tests/test_cpp_headers.py compiles them there).
  typedef Eigen::Matrix<double, 6, 1> EVector6d;
  typedef Eigen::Matrix<double, 6, Eigen::Dynamic> EMatrix6Xd;
  typedef std::vector<Eigen::Affine3d, Eigen::aligned_allocator<Eigen::Affine3d>> EVectorOfAffine3d;   // internal/types.h:137
  typedef std::vector<EVector6d, Eigen::aligned_allocator<EVector6d>> EVectorOfVector6d;                 // internal/types.h:138

  Eigen::Affine3d getTransformation(const Eigen::VectorXd& q) { return eAffine(getTransformation(stdv(q))); }
  EVectorOfAffine3d getTransformations(const Eigen::VectorXd& q)
  {
    const std::vector<Affine3dImage> t = getTransformations(stdv(q));
    EVectorOfAffine3d out;
    for (const Affine3dImage& a : t) out.push_back(eAffine(a));
    return out;
  }
  EMatrix6Xd getJacobian(const Eigen::VectorXd& q)
  {
    const VectorXd j = getJacobian(stdv(q));
    EMatrix6Xd J(6, (int)m_n);
    for (unsigned c = 0; c < m_n; c++)
      for (int r = 0; r < 6; r++) J(r, c) = j[6 * c + r];
    return J;
  }
  EVectorOfVector6d getTwist(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq) { return eSix(getTwist(stdv(q), stdv(Dq))); }
  EVector6d getTwistTool(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq) { return getTwist(q, Dq).back(); }
  EVectorOfVector6d getDTwist(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq, const Eigen::VectorXd& DDq)
  {
    return eSix(getDTwist(stdv(q), stdv(Dq), stdv(DDq)));
  }
  EVector6d getDTwistTool(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq, const Eigen::VectorXd& DDq) { return getDTwist(q, Dq, DDq).back(); }
  EVectorOfVector6d getDTwistLinearPart(const Eigen::VectorXd& q, const Eigen::VectorXd& DDq) { return eSix(getDTwistLinearPart(stdv(q), stdv(DDq))); }
  EVectorOfVector6d getDTwistNonLinearPart(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq) { return eSix(getDTwistNonLinearPart(stdv(q), stdv(Dq))); }
  EVectorOfVector6d getDDTwist(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq, const Eigen::VectorXd& DDq, const Eigen::VectorXd& DDDq)
  {
    return eSix(getDDTwist(stdv(q), stdv(Dq), stdv(DDq), stdv(DDDq)));
  }
  EVector6d getDDTwistTool(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq, const Eigen::VectorXd& DDq, const Eigen::VectorXd& DDDq)
  {
    return getDDTwist(q, Dq, DDq, DDDq).back();
  }
  EVectorOfVector6d getDDTwistLinearPart(const Eigen::VectorXd& q, const Eigen::VectorXd& DDDq) { return eSix(getDDTwistLinearPart(stdv(q), stdv(DDDq))); }
  EVectorOfVector6d getDDTwistNonLinearPart(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq, const Eigen::VectorXd& DDq)
  {
    return eSix(getDDTwistNonLinearPart(stdv(q), stdv(Dq), stdv(DDq)));
  }
  Eigen::VectorXd getJointTorque(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq, const Eigen::VectorXd& DDq)
  {
    return eVec(getJointTorque(stdv(q), stdv(Dq), stdv(DDq)));
  }
  Eigen::VectorXd getJointTorqueNonLinearPart(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq) { return eVec(getJointTorqueNonLinearPart(stdv(q), stdv(Dq))); }
  Eigen::MatrixXd getRegressor(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq, const Eigen::VectorXd& DDq)
  {
    return eMat(getRegressor(stdv(q), stdv(Dq), stdv(DDq)), (int)m_n, (int)(10 * m_nj));
  }
  Eigen::MatrixXd getJointInertia(const Eigen::VectorXd& q) { return eMat(getJointInertia(stdv(q)), (int)m_n, (int)m_n); }
  Eigen::VectorXd getJointAcceleration(const Eigen::VectorXd& q, const Eigen::VectorXd& Dq, const Eigen::VectorXd& tau)
  {
    return eVec(getJointAcceleration(stdv(q), stdv(Dq), stdv(tau)));
  }
  Eigen::VectorXd getNominalParametersEigen() const { return eVec(getNominalParameters()); }

  // Batched siblings for Eigen callers: N samples as the COLUMNS of n_act x N matrices (column-major, i.e. one sample = n_act contiguous
  // doubles); results come back in the Eigen-record layout (RDB_LAYOUT_EIGEN), so sample i of the regressor is the contiguous column-major
  // n_act x 10 nJ block at out.data() + i * n_act * 10 nJ -- a plain Eigen::Map<const Eigen::MatrixXd> views it.
  // (AoS inputs are transposed into SoA planes on the host first; identification data kept as SoA from the start skips that copy through the
  // rdb_samples overloads above.)
  void getRegressorBatch(const Eigen::MatrixXd& q, const Eigen::MatrixXd& Dq, const Eigen::MatrixXd& DDq, std::vector<double>& regressor_records,
                         std::vector<double>* torque_records = nullptr)
  {
    if (q.rows() != (int)m_n || Dq.rows() != q.rows() || DDq.rows() != q.rows() || Dq.cols() != q.cols() || DDq.cols() != q.cols())
      throw std::invalid_argument("Input data dimensions mismatch");
    const int64_t n = (int64_t)q.cols();
    const VectorXd sq = soa(q), sdq = soa(Dq), sddq = soa(DDq);
    regressor_records.resize((size_t)n * m_n * 10 * m_nj);
    if (torque_records) torque_records->resize((size_t)n * m_n);
    rdb_samples in{n, n > 0 ? n : 1, sq.data(), sdq.data(), sddq.data(), nullptr};
    rdb_dynamics_out out{};
    out.ld = in.ld;
    out.layout = RDB_LAYOUT_EIGEN;
    out.regressor = regressor_records.data();
    out.torque = torque_records ? torque_records->data() : nullptr;
    check(rdb_dynamics_batch_host(m_h, &in, &out));
  }
#endif

private:
  rdb_chain* m_h = nullptr;
  unsigned int m_nj = 0, m_nl = 0, m_n = 0;

  static void check(rdb_status s)
  {
    if (s == RDB_OK) return;
    if (s == RDB_ERR_DIM_MISMATCH || s == RDB_ERR_INVALID_ARG) throw std::invalid_argument(rdb_last_error());
    throw std::runtime_error(std::string("rosdyn_b200: ") + rdb_last_error());
  }
  void sizes(const VectorXd& q, const VectorXd* a, const VectorXd* b, const VectorXd* c) const
  {
    if (q.size() != m_n || (a && a->size() != m_n) || (b && b->size() != m_n) || (c && c->size() != m_n))
      throw std::invalid_argument("Input data dimensions mismatch");
  }
  VectorXd kin1(const VectorXd& q, const VectorXd* Dq, const VectorXd* DDq, const VectorXd* DDDq, double* rdb_kinematics_out::*field, size_t rows,
                int32_t layout = RDB_LAYOUT_SOA)
  {
    sizes(q, Dq, DDq, DDDq);
    VectorXd out(rows);
    rdb_samples in{1, 1, q.data(), Dq ? Dq->data() : nullptr, DDq ? DDq->data() : nullptr, DDDq ? DDDq->data() : nullptr};
    rdb_kinematics_out o{};
    o.ld = 1;
    o.layout = layout;
    o.*field = out.data();
    check(rdb_kinematics_batch_host(m_h, &in, &o));
    return out;
  }
#ifdef ROSDYN_B200_HAVE_EIGEN
  static VectorXd stdv(const Eigen::VectorXd& v)
  {
    VectorXd o((size_t)v.size());
    for (size_t k = 0; k < o.size(); k++) o[k] = v((int)k);
    return o;
  }
  static Eigen::VectorXd eVec(const VectorXd& v)
  {
    Eigen::VectorXd o((int)v.size());
    for (size_t k = 0; k < v.size(); k++) o((int)k) = v[k];
    return o;
  }
  static Eigen::MatrixXd eMat(const VectorXd& v, int rows, int cols)  // column-major image -> matrix
  {
    Eigen::MatrixXd o(rows, cols);
    for (int c = 0; c < cols; c++)
      for (int r = 0; r < rows; r++) o(r, c) = v[(size_t)c * rows + r];
    return o;
  }
  static Eigen::Affine3d eAffine(const Affine3dImage& a)
  {
    Eigen::Affine3d T;
    for (int c = 0; c < 4; c++)
      for (int r = 0; r < 4; r++) T.matrix()(r, c) = a[4 * c + r];
    return T;
  }
  static EVectorOfVector6d eSix(const std::vector<Vector6d>& v)
  {
    EVectorOfVector6d o(v.size());
    for (size_t l = 0; l < v.size(); l++)
      for (int k = 0; k < 6; k++) o[l](k) = v[l][k];
    return o;
  }
  static VectorXd soa(const Eigen::MatrixXd& x)  // n_act x N (samples as columns) -> SoA planes x[joint][N]
  {
    const int64_t rows = x.rows(), cols = x.cols();
    VectorXd o((size_t)(rows * cols));
    for (int64_t r = 0; r < rows; r++)
      for (int64_t c = 0; c < cols; c++) o[(size_t)(r * cols + c)] = x((int)r, (int)c);
    return o;
  }
#endif
  static std::vector<Vector6d> six(const VectorXd& v)
  {
    std::vector<Vector6d> out(v.size() / 6);
    for (size_t l = 0; l < out.size(); l++)
      for (int k = 0; k < 6; k++) out[l][k] = v[6 * l + k];
    return out;
  }
};

}  // namespace rosdyn_b200

#ifdef ROSDYN_B200_DROP_IN
namespace rosdyn = rosdyn_b200;  // lets `rosdyn::Chain` in identification code name this class
#endif

#endif  // ROSDYN_B200_CHAIN_HPP
