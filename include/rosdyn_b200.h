/*
 * rosdyn_b200.h -- C-ABI of the B200-native batched chain-dynamics engine.
 *
 * Drop-in boundary for the hot path of rosdyn_core's `rosdyn::Chain`
 * (reference: rosdyn_core/include/rosdyn_core/primitives.h:235-555, implementation
 * rosdyn_core/include/rosdyn_core/internal/primitives_impl.h:863-1391; abbreviated P.h / PI.h below).
 * The reference has no FFI today (header-only C++ on Eigen); this is the set of entry points a
 * reference-side binding would call instead of looping `Chain::get*` once per sample.
 *
 * Conventions (all mirrored from the reference, see SURVEY.md appendix A):
 *   - plain C types only; every entry returns an int32 status, never throws;
 *   - the caller owns every buffer; the library owns only the opaque handle and its device workspace;
 *   - batched arrays are SoA "planes": x[component][ld] with `ld >= n` samples, fp64;
 *   - joint vectors q/Dq/DDq/DDDq have one plane per INPUT joint (input order, `S` of PI.h:708-731);
 *   - 6-vectors are [linear(3); angular(3)] (spacevect_algebra.h:44-53), one block of 6 planes per link,
 *     link 0 = base (always zero, PI.h:661-677);
 *   - poses are 3x4 [R|p] row-major: plane r*4+c;
 *   - matrices that the reference returns as Eigen column-major (Jacobian 6 x n, regressor n x 10*nJ,
 *     inertia n x n) use plane index  col*rows + row;
 *   - every batched evaluation is STATELESS: each sample is a fresh evaluation through the reference's
 *     direct path (the reference's dirty-flag caches, PI.h:886/985/1088, are not reproduced);
 *   - `stream` is a cudaStream_t passed as void*; device entry points are asynchronous on it;
 *   - a handle lives on ONE device (the current device at rdb_chain_create, or the one given to rdb_chain_create_on); every entry point
 *     makes that device current for the call and restores the caller's device, so handles of several devices can be driven from one thread;
 *   - entries that take `const rdb_chain*` only read the handle and may run concurrently on one handle (distinct streams); entries that take
 *     `rdb_chain*` use per-handle workspaces and are serialised by a per-handle lock.
 *
 * There is no CPU fallback: every compute entry fails with RDB_ERR_NO_DEVICE when no CUDA device exists.
 */
#ifndef ROSDYN_B200_H
#define ROSDYN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RDB_ABI_VERSION 2
#define RDB_MAX_JOINTS 64 /* chain joints incl. fixed (reference: NUM_MAX_AXES 40, internal/types.h:126) */

typedef int32_t rdb_status;
enum
{
  RDB_OK = 0,
  RDB_ERR_INVALID_ARG = 1,  /* null pointer, bad size, malformed descriptor                                  */
  RDB_ERR_DIM_MISMATCH = 2, /* q/Dq/DDq not all present  (PI.h:1299-1309 throws std::invalid_argument)        */
  RDB_ERR_CUDA = 3,         /* a CUDA runtime call failed; see rdb_last_error()                               */
  RDB_ERR_NO_DEVICE = 4,    /* no CUDA device: the product path has no CPU fallback                           */
  RDB_ERR_NOT_FOUND = 5,    /* "Base link not found"/"Tool link not found"/unknown link (PI.h:601-613,918-921) */
  RDB_ERR_ALLOC = 6
};

enum
{
  RDB_JOINT_FIXED = 0,    /* rosdyn::Joint::FIXED,     T_pc = T_pj                               (PI.h:82-83) */
  RDB_JOINT_REVOLUTE = 1, /* REVOLUTE and URDF continuous, R_jc = I + sin q K + (1-cos q) K^2    (PI.h:40-44) */
  RDB_JOINT_PRISMATIC = 2 /* PRISMATIC, t = t_pj + axis_p q                                      (PI.h:45-46) */
};

/* One chain joint, as Joint::fromUrdf leaves it (PI.h:50-83). */
typedef struct rdb_joint_desc
{
  int32_t type;        /* RDB_JOINT_*                                                                      */
  int32_t input_index; /* position of this joint in q/Dq/DDq (column of S, PI.h:728), or -1: q == 0        */
  double xyz[3];       /* parent->joint origin translation  t_pj                                            */
  double rot[9];       /* parent->joint origin rotation R_pj, row-major (URDF rpy: Rz(y) Ry(p) Rx(r))       */
  double axis[3];      /* joint axis in the joint frame; normalised on create when non-zero (PI.h:58-59)    */
} rdb_joint_desc;

/* One chain link, as Link::fromUrdf reads it (PI.h:288-319). */
typedef struct rdb_link_desc
{
  double mass;
  double cog[3];          /* inertial origin xyz in the link frame                                          */
  double inertial_rot[9]; /* inertial-frame rotation R_p_cog, row-major (identity when rpy == 0)            */
  double inertia[6];      /* ixx ixy ixz iyy iyz izz about the cog, in the inertial frame                   */
} rdb_link_desc;

/* A serial chain base->tool: n_joints joints (fixed ones INCLUDED, PI.h:638) and n_joints+1 links. */
typedef struct rdb_chain_desc
{
  int32_t n_joints;
  int32_t n_inputs; /* length of the joint vectors = number of input joints (PI.h:739)                      */
  double gravity[3];
  const rdb_joint_desc* joints; /* [n_joints], base -> tool                                                */
  const rdb_link_desc* links;   /* [n_joints + 1], links[0] = base link (its inertia is never used)        */
} rdb_chain_desc;

typedef struct rdb_chain rdb_chain; /* opaque */

/* ---- library ------------------------------------------------------------------------------------- */
int32_t rdb_abi_version(void);
const char* rdb_last_error(void);       /* thread-local text of the last failure                            */
const char* rdb_status_string(rdb_status s);
int32_t rdb_device_count(void);         /* 0 when no CUDA device / driver                                   */
uint64_t rdb_kernel_launch_count(void); /* kernels launched by this library since load (bench evidence)     */

/* ---- chain handle (replaces rosdyn::createChain / Chain::init, PI.h:580-703, 1518-1527) ----------- */
rdb_status rdb_chain_create(const rdb_chain_desc* desc, rdb_chain** out);
void rdb_chain_destroy(rdb_chain* chain);
/* Chain::setInputJointsName by index (PI.h:705-742): chain_joint_of_input[i] = chain joint fed by input i. */
rdb_status rdb_chain_set_input_joints(rdb_chain* chain, int32_t n_inputs, const int32_t* chain_joint_of_input);
int32_t rdb_chain_joints_number(const rdb_chain* chain);        /* Chain::getJointsNumber       P.h:381   */
int32_t rdb_chain_links_number(const rdb_chain* chain);         /* Chain::getLinksNumber        P.h:377   */
int32_t rdb_chain_active_joints_number(const rdb_chain* chain); /* Chain::getActiveJointsNumber P.h:385   */
rdb_status rdb_chain_gravity(const rdb_chain* chain, double out[3]); /* Chain::getGravity P.h:409          */
/* Chain::getNominalParameters (PI.h:1382-1391): out[10*n_joints], per link m, mcx,mcy,mcz, Ixx,Ixy,Ixz,Iyy,Iyz,Izz */
rdb_status rdb_chain_nominal_parameters(const rdb_chain* chain, double* out);

/* ---- URDF -> chain (replaces urdfdom + Link/Joint::fromUrdf + Chain::init, PI.h:50-149, 276-331, 580-703) ---- */
/* The chain between base_link and tool_link of a URDF document, as the reference would extract it.  Owned by the
 * library; `desc` and every array stay valid until rdb_urdf_chain_free.  Limits follow PI.h:85-143 (malformed-URDF
 * defaults included); default inputs are the moveable joints base -> tool (PI.h:631-636, 700). */
typedef struct rdb_urdf_chain
{
  rdb_chain_desc desc;
  const char* const* joint_names; /* [n_joints]      */
  const char* const* link_names;  /* [n_joints + 1]  */
  const double* q_max;            /* [n_joints] per chain joint (0 for fixed joints) */
  const double* q_min;
  const double* dq_max;
  const double* ddq_max;
  const double* tau_max;
} rdb_urdf_chain;
/* RDB_ERR_NOT_FOUND + "Base link not found" / "Tool link not found" (PI.h:601-613); gravity NULL = zero (P.h:346). */
rdb_status rdb_urdf_parse(const char* urdf_xml, const char* base_link, const char* tool_link, const double gravity[3], rdb_urdf_chain** out);
void rdb_urdf_chain_free(rdb_urdf_chain* chain);
/* rosdyn::createChain(model, base, tool, gravity) (PI.h:1518-1527): parse + rdb_chain_create. */
rdb_status rdb_chain_from_urdf(const char* urdf_xml, const char* base_link, const char* tool_link, const double gravity[3], rdb_chain** out);

/* ---- batched inputs ------------------------------------------------------------------------------ */
typedef struct rdb_samples
{
  int64_t n;          /* number of samples                                                                 */
  int64_t ld;         /* plane stride (doubles), ld >= n                                                   */
  const double* q;    /* [n_inputs][ld]                                                                    */
  const double* dq;   /* [n_inputs][ld] or NULL (== 0)                                                     */
  const double* ddq;  /* [n_inputs][ld] or NULL (== 0, e.g. getJointTorqueNonLinearPart PI.h:1285-1293)    */
  const double* dddq; /* [n_inputs][ld] or NULL (== 0)                                                     */
} rdb_samples;

/* Output layout of the batched entries that have a `layout` selector (reference containers: internal/types.h:137-141).
 *   RDB_LAYOUT_SOA   : SoA planes x[component][ld] as described at the top of this file (the fast layout: coalesced stores).
 *   RDB_LAYOUT_EIGEN : one dense record per sample, laid out exactly as the reference's Eigen object lies in memory, so a host
 *                      (or device) `Eigen::Map` can view sample i at  base + i * record  with no conversion; `ld` is ignored:
 *       poses       Eigen::Affine3d image: 16 doubles, 4x4 COLUMN-major incl. the [0 0 0 1] row; T_tool[n][16],
 *                   T_links[n][nL][16] (= the storage of a VectorOfAffine3d, T.h:137)
 *       6-vectors   [n][nL][6]                      (= VectorOfVector6d, T.h:138)
 *       jacobian    [n][6 * n_inputs]   column-major 6 x n_inputs   (Matrix6Xd)
 *       regressor   [n][n_inputs * 10 * n_joints] column-major n_inputs x 10 n_joints (Eigen::MatrixXd as getRegressor returns it)
 *       inertia     [n][n_inputs * n_inputs], torque [n][n_inputs]
 *     One record per sample: the regressor records of a warp are staged in shared memory and written row-wise (0.43 of the HBM peak against
 *     0.96 for the SoA planes, DESIGN.md 3.1); the other outputs are stored per thread.  For a host consumer the records come back with ONE
 *     contiguous copy per chunk instead of one strided copy per plane. */
enum
{
  RDB_LAYOUT_SOA = 0,
  RDB_LAYOUT_EIGEN = 1
};

/* Kinematics outputs; every pointer is optional (NULL = not produced). nL = n_joints + 1.  Zero-initialise the struct: `layout` = 0 is SoA. */
typedef struct rdb_kinematics_out
{
  int64_t ld;             /* plane stride of every output below, ld >= n  (RDB_LAYOUT_SOA)                  */
  double* T_tool;         /* [12][ld]        Chain::getTransformation            PI.h:884                   */
  double* T_links;        /* [nL][12][ld]    Chain::getTransformations           PI.h:908                   */
  double* jacobian;       /* [n_inputs*6][ld] Chain::getJacobian, plane col*6+row PI.h:927                  */
  double* twist;          /* [nL][6][ld]     Chain::getTwist                     PI.h:981                   */
  double* dtwist;         /* [nL][6][ld]     Chain::getDTwist                    PI.h:1082 (direct path)    */
  double* dtwist_lin;     /* [nL][6][ld]     Chain::getDTwistLinearPart          PI.h:1029                  */
  double* dtwist_nonlin;  /* [nL][6][ld]     Chain::getDTwistNonLinearPart       PI.h:1063                  */
  double* ddtwist;        /* [nL][6][ld]     Chain::getDDTwist                   PI.h:1185 (direct path)    */
  double* ddtwist_lin;    /* [nL][6][ld]     Chain::getDDTwistLinearPart         PI.h:1126 (correct buffer) */
  double* ddtwist_nonlin; /* [nL][6][ld]     Chain::getDDTwistNonLinearPart      PI.h:1156                  */
  double* torque;         /* [n_inputs][ld]  Chain::getJointTorque (no ext. wrench) PI.h:1277               */
  int32_t layout;         /* RDB_LAYOUT_SOA (0) or RDB_LAYOUT_EIGEN: shapes above become the per-sample records */
} rdb_kinematics_out;

/* Dynamics outputs of rdb_dynamics_batch; every pointer is optional.  P = 10 * n_joints. */
typedef struct rdb_dynamics_out
{
  int64_t ld;        /* plane stride (RDB_LAYOUT_SOA), ld >= n                                                      */
  double* regressor; /* [P * n_inputs][ld], plane col*n_inputs+row   Chain::getRegressor      PI.h:1295            */
  double* torque;    /* [n_inputs][ld]                               Chain::getJointTorque    PI.h:1277            */
  double* inertia;   /* [n_inputs * n_inputs][ld], plane col*n_inputs+row  Chain::getJointInertia PI.h:1357        */
  int32_t layout;    /* RDB_LAYOUT_SOA (0) or RDB_LAYOUT_EIGEN                                                      */
} rdb_dynamics_out;

/* ---- batched device entry points (pointers are DEVICE pointers) ----------------------------------- */
/* FK, Jacobian, twist / acceleration / jerk recursions and RNEA torque in one pass over the chain. */
rdb_status rdb_kinematics_batch(const rdb_chain* chain, const rdb_samples* in, const rdb_kinematics_out* out, void* stream);

/* Chain::getJointTorque(q,Dq,DDq) (PI.h:1277-1283): torque[n_inputs][ld_out]. */
rdb_status rdb_torque_batch(const rdb_chain* chain, const rdb_samples* in, double* torque, int64_t ld_out, void* stream);

/* Chain::getRegressor (PI.h:1295-1355): phi[(10*n_joints)*n_inputs][ld_out], plane col*n_inputs+row, every
 * plane written (structural zeros are exact 0.0).  `torque` optional: getJointTorque of the same samples. */
rdb_status rdb_regressor_batch(const rdb_chain* chain, const rdb_samples* in, double* phi, double* torque, int64_t ld_out, void* stream);

/* Chain::getJointInertia (PI.h:1357-1379): inertia[n_inputs*n_inputs][ld_out], plane col*n_inputs+row. */
rdb_status rdb_inertia_batch(const rdb_chain* chain, const rdb_samples* in, double* inertia, int64_t ld_out, void* stream);

/* getRegressor / getJointTorque / getJointInertia of the same samples with a selectable output layout (the three entries above are the
 * SoA special cases).  Regressor and torque come from one pass over the chain, the inertia from a second launch. */
rdb_status rdb_dynamics_batch(const rdb_chain* chain, const rdb_samples* in, const rdb_dynamics_out* out, void* stream);

/* Forward dynamics (no reference function; the reference's callers compose getJointInertia PI.h:1357-1379 and
 * getJointTorqueNonLinearPart PI.h:1285-1293):  ddq = M(q)^-1 (tau - h(q, Dq)),  h = getJointTorque(q, Dq, 0) incl. gravity.
 * in->q, in->dq (NULL = 0) as everywhere; in->ddq / in->dddq are ignored.  tau[n_inputs][in->ld] (NULL = zero torque, the same
 * plane stride as q, like tau_meas of rdb_regressor_gram_batch).  ddq[n_inputs][ld_out].  info[n] optional: 0, or 1 when M(q) is not
 * positive definite (a Cholesky pivot <= 0 or not finite); that sample's ddq is NaN in every component.
 * Inputs that no chain joint feeds get ddq = 0 and are left out of the solve (their row / column of M is zero).
 * One pass over the chain per sample: M and h are accumulated in registers, M is factored there (Cholesky) and only ddq leaves the
 * thread.  Results are per sample: bit-identical across launches and between this entry and its host twin.
 * Additive joint components (friction, springs) compose by subtraction: copy tau, then
 * rdb_components_torque_batch(chain, in, -pi_c, tau_copy, ld, accumulate = 1, stream) adds -Phi_c pi_c, and forward dynamics of tau_copy
 * gives M^-1 (tau - h - Phi_c pi_c). */
rdb_status rdb_forward_dynamics_batch(const rdb_chain* chain, const rdb_samples* in, const double* tau, double* ddq, int64_t ld_out,
                                      int32_t* info, void* stream);

/* Fused regressor -> normal equations (no reference code: the consumer rosdyn_identification is external,
 * reference README.md:15).  With P = 10*n_joints and Phi_s the n_inputs x P regressor of sample s:
 *   gram[P*P]  (+)= sum_s Phi_s^T Phi_s   (column-major, full symmetric matrix)
 *   rhs[P]     (+)= sum_s Phi_s^T tau_s
 *   tau_sq[1]  (+)= sum_s tau_s^T tau_s
 * tau_s = tau_meas[n_inputs][ld] when given, else getJointTorque(q,Dq,DDq) of the sample.
 * accumulate != 0 adds to the existing contents of gram/rhs/tau_sq (chunked / resumable use). */
rdb_status rdb_regressor_gram_batch(rdb_chain* chain, const rdb_samples* in, const double* tau_meas, double* gram, double* rhs,
                                    double* tau_sq, int32_t accumulate, void* stream);

/* Chain::getWrench / Chain::getJointTorque(q,Dq,DDq,ext_wrenches_in_link_frame) (PI.h:1225-1274).
 * ext_wrenches[nL][6][ld_ext]: wrenches applied TO the links, in link frames, [force; torque] per link (NULL = none).  The reference
 * brings them to the base frame with the TWIST transform spatialTranformation(-ext, T_bl) (PI.h:1255, SA.h:193-197); mirrored
 * literally.  Outputs (each optional): torque[n_inputs][ld_out]; wrenches[nL][6][ld_out] = m_wrenches (base frame, at each link
 * origin, link 0 included). */
rdb_status rdb_wrench_batch(const rdb_chain* chain, const rdb_samples* in, const double* ext_wrenches, int64_t ld_ext, double* torque,
                            double* wrenches, int64_t ld_out, void* stream);
/* Chain::getJacobianLink(q, link) (PI.h:951-979): jacobian[n_inputs*6][ld_out], plane col*6+row, of link `link_index`
 * (0 = base ... n_joints = tool), evaluated at q.  As in the reference the first K input joints get a column, K = number of
 * input joints between the base and the link (the reference indexes m_active_joints by the loop counter, PI.h:970); with the
 * default base->tool input order those are exactly the joints that move the link.  RDB_ERR_NOT_FOUND for a link outside the
 * chain ("link ... is not member of the chain", PI.h:960). */
rdb_status rdb_jacobian_link_batch(const rdb_chain* chain, const rdb_samples* in, int32_t link_index, double* jacobian, int64_t ld_out,
                                   void* stream);

/* Chain::computeLocalIk / computeWeigthedLocalIk (PI.h:1398-1468), batched: for every target pose, Gauss-Newton steps
 *   dq = argmin |J dq - e|^2_W  s.t.  q_min <= sol + dq <= q_max,   e = getFrameDistance(T_target, T(sol))  (frame_distance.h:44-49)
 * from `seed` until |W e| < toll.  The reference's wall-clock budget (ros::Duration max_time) becomes an ITERATION budget `max_iter`
 * (at most max_iter steps, max_iter + 1 convergence checks) and Eigen::solve_quadprog of the un-vendored eigen_matrix_utils becomes an exact
 * box-constrained active-set solve.  target[12][ld]: 3x4 [R|p] row-major planes (the layout of rdb_kinematics_out.T_tool);
 * seed / sol [n_inputs][ld]; q_min / q_max [n_inputs] HOST arrays (NULL = -/+1e10, the reference's no-limit default, PI.h:92-93);
 * weight[6] host array or NULL (NULL = computeLocalIk).  Optional outputs: status[n] (1 = converged, the reference's return value),
 * iterations[n], error_norm[n] (|W e| at return).  n_inputs <= RDB_IK_MAX_INPUTS. */
#define RDB_IK_MAX_INPUTS 8
rdb_status rdb_local_ik_batch(const rdb_chain* chain, int64_t n, int64_t ld, const double* target, const double* seed, const double* q_min,
                              const double* q_max, const double* weight, double toll, int32_t max_iter, double* sol, int32_t* status,
                              int32_t* iterations, double* error_norm, void* stream);

/* ---- additive joint components (SURVEY.md section 8f N2) ------------------------------------------------------------
 * The reference models joint friction / elasticity as per-joint "components" whose regressor columns are appended to the
 * inertial regressor by the identification code (base_component.h:124-139).  Column blocks, in the order given here:
 *   RDB_COMPONENT_FRICTION_POLY1 (FirstOrderPolynomialFriction, friction_polynomial1.h:45-52):   [sign, omega]
 *        omega = clamp(Dq_j, -max_velocity, max_velocity), sign = clamp(omega / min_velocity, -1, 1)
 *   RDB_COMPONENT_FRICTION_POLY2 (SecondOrderPolynomialFriction, friction_polynomial2.h:42-58):  [sign, omega, omega^2 sign]
 *        sign = 0 (omega == 0), +-1 beyond +-min_velocity, omega / min_velocity in between
 *   RDB_COMPONENT_IDEAL_SPRING   (IdealSpring, ideal_spring.h:64-70):                            [q_j, 1]
 * Constructor rules are mirrored: min_velocity < 1e-6 becomes 1e-6; POLY1 max_velocity <= 0 becomes 1e6
 * (friction_polynomial1.h:74-87); POLY2 with max_velocity < 0 sets min_velocity = 1e6 and keeps max_velocity, as the
 * reference does (friction_polynomial2.h:91-96).  Every column is zero except in the row of its joint. */
typedef enum rdb_component_type
{
  RDB_COMPONENT_FRICTION_POLY1 = 1,
  RDB_COMPONENT_FRICTION_POLY2 = 2,
  RDB_COMPONENT_IDEAL_SPRING = 3
} rdb_component_type;
#define RDB_MAX_COMPONENTS 64
typedef struct rdb_component_desc
{
  int32_t type;        /* rdb_component_type                                                                */
  int32_t input_index; /* the joint it acts on, as a position in q/Dq (ComponentBase::getJointNumber)       */
  double min_velocity; /* friction constants "min_velocity" / "max_velocity"; ignored by the spring         */
  double max_velocity;
} rdb_component_desc;
int32_t rdb_component_columns(int32_t type); /* 2, 3, 2; -1 for an unknown type (ComponentBase::getParametersNumber) */
/* n = 0 clears.  rdb_chain_set_input_joints DROPS the components (their input_index refers to the old input vector): set them again. */
rdb_status rdb_chain_set_components(rdb_chain* chain, int32_t n, const rdb_component_desc* components);
int32_t rdb_chain_component_columns(const rdb_chain* chain); /* total number of component columns Pc */
/* ComponentBase::getRegressor of every component, side by side: phi_c[Pc * n_inputs][ld_out], plane col*n_inputs+row. */
rdb_status rdb_components_regressor_batch(const rdb_chain* chain, const rdb_samples* in, double* phi_c, int64_t ld_out, void* stream);
/* ComponentBase::getTorque summed over the components: torque[n_inputs][ld_out] (+)= phi_c(sample) * parameters;
 * parameters[Pc] is a HOST array (the components' nominal parameters).  IdealSpring::getTorque indexes q out of range in
 * the reference (ideal_spring.h:57); this entry uses regressor * parameters, the evident intent. */
rdb_status rdb_components_torque_batch(const rdb_chain* chain, const rdb_samples* in, const double* parameters, double* torque,
                                       int64_t ld_out, int32_t accumulate, void* stream);
/* Normal equations of the extended model [Phi | Phi_c] with Pt = 10*n_joints + Pc columns: gram[Pt*Pt], rhs[Pt], tau_sq[1];
 * same conventions as rdb_regressor_gram_batch.  tau_s = tau_meas when given, else the rigid-body getJointTorque. */
rdb_status rdb_regressor_gram_ext_batch(rdb_chain* chain, const rdb_samples* in, const double* tau_meas, double* gram, double* rhs,
                                        double* tau_sq, int32_t accumulate, void* stream);

/* Chain::getMultiplicity (PI.h:1470-1517), HOST arrays: every joint vector q + 2 pi k that stays inside [q_min, q_max], revolute input
 * joints only (joint_type_of_input[i] = RDB_JOINT_* of the chain joint fed by input i), in the reference's order (q first; per joint
 * the positive turns, then the negative ones; joints combined base -> tool).  out[count][n_inputs] row-major; *count is always set to the
 * number of vectors; RDB_ERR_INVALID_ARG when capacity is too small (nothing beyond capacity is written) or when a revolute joint's limits
 * span more than 1000 turns (the reference would enumerate them all). */
rdb_status rdb_multiplicity(int32_t n_inputs, const int32_t* joint_type_of_input, const double* q, const double* q_min, const double* q_max,
                            double* out, int64_t capacity, int64_t* count);

/* Host-only utility (used by the tests): the constant 10x10 map T = d(parameters referred to frame A) / d(parameters referred to frame B)
 * of a body rigidly attached with x_A = R x_B + t (R row-major), T[c * 10 + p], parameters [m, m c, Ixx, Ixy, Ixz, Iyy, Iyz, Izz] about
 * the frame origin (PI.h:399-417).  It is what folds never-moving joints out of the chain for the fused normal equations, the torque and
 * the inertia walkers: Phi[:, block B] = Phi[:, block A] T. */
rdb_status rdb_fold_parameter_map(const double* R, const double* t, double* T);

/* Host-only utility (used by the tests): the rotation Q (row-major, det +1) with Q e_z = axis that turns the frame of a revolute link of the
 * folded chain, x_old = Q x_new, so that its joint axis is e_z.  An axis along a coordinate axis gets an exact signed permutation matrix.
 * RDB_ERR_INVALID_ARG when axis is not a unit vector. */
rdb_status rdb_fold_canonical_frame(const double* axis, double* Q);

/* Host-only utility (used by the tests): the row layout of the fused normal-equation kernel on all-revolute folded chains of nj (1..7) moving
 * joints.  pos[j * 10 nj + c]: the position of parameter column c inside the kernel's row of joint j, or -1 where the row stores nothing (the
 * blocks of the links before j, and the columns the all-revolute regressor makes exact zeros); rowlen[j]: the positions of that row;
 * *tau_col: 1 when tau is position 0 of every row, 0 when it is accumulated beside the tiles.  RDB_ERR_INVALID_ARG for other nj. */
rdb_status rdb_gram_row_layout(int32_t nj, int32_t* pos, int32_t* rowlen, int32_t* tau_col);

/* ---- normal-equation solve (SURVEY.md section 8f N3; HOST arrays, no reference code: the consumer is external) ------
 * Minimum-norm least-squares solution of gram * parameters = rhs through a symmetric eigen-decomposition: the regressor is rank
 * deficient in the standard parameters, so eigenvalues <= rel_tol * lambda_max (rel_tol <= 0: 1e-10) are discarded.
 * gram[P*P] column-major (as rdb_regressor_gram_batch returns it, copied to the host), rhs[P]; outputs parameters[P],
 * optional eigenvalues[P] (descending), rank, residual_sq = tau_sq - 2 pi^T rhs + pi^T gram pi = sum ||Phi pi - tau||^2. */
rdb_status rdb_normal_equations_solve(int32_t P, const double* gram, const double* rhs, double tau_sq, double rel_tol, double* parameters,
                                      double* eigenvalues, int32_t* rank, double* residual_sq);

/* ---- one process, several GPUs (SURVEY.md section 8e) ---------------------------------------------------------------
 * rdb_chain_create uses the CURRENT device; rdb_chain_create_on creates the handle on `device` (and restores the current device).
 * rdb_regressor_gram_sharded_host: samples are independent, so the HOST batch is cut into n_chains contiguous shards
 * [r n / R, (r+1) n / R), shard r runs through rdb_regressor_gram_batch_host on chains[r] (its device; one worker thread per handle, all
 * concurrently), and the R partial normal equations are summed on the host in rank order -- bit-reproducible for a given R, no collective
 * library needed.  The handles must describe the same chain (same joints / inputs); several handles may share a device. */
rdb_status rdb_chain_create_on(const rdb_chain_desc* desc, int32_t device, rdb_chain** out);
int32_t rdb_chain_device(const rdb_chain* chain);
/* Which normal-equation kernel the chain's last rdb_regressor_gram* call ran: *specialised = 1 for the fused kernel compiled at run time
 * (NVRTC) against the chain's own constants, 0 for the precompiled fused kernel (chains that are not all-revolute, NVRTC missing or failing,
 * RDB_GRAM_JIT=0), 2 for the general pipeline (materialised regressor and tiled contraction: more than 7 moving joints, no moving joint, or
 * a component set the one-pass kernel refuses), -1 before the first call.  reason (optional, reason_len bytes, NUL-terminated) says why, or
 * how long the compile took; for the general pipeline it starts with "general pipeline:". */
rdb_status rdb_chain_gram_kernel_info(const rdb_chain* chain, int32_t* specialised, char* reason, int32_t reason_len);
/* Host only, no device needed (inspection tools): the cubin of the run-time specialised kernel of an all-revolute chain, written to `path`.
 * kernel_args: the kernel and its template arguments without the model, e.g. "gram_fused_kernel<6, 4, true, 0"; arch e.g. "sm_100a". */
rdb_status rdb_gram_specialised_cubin(const rdb_chain_desc* desc, const char* kernel_args, const char* arch, const char* path, char* reason,
                                      int32_t reason_len);
rdb_status rdb_regressor_gram_sharded_host(rdb_chain* const* chains, int32_t n_chains, const rdb_samples* in, const double* tau_meas,
                                           double* gram, double* rhs, double* tau_sq, int32_t accumulate);

/* ---- several GPUs over NVLink: the sharded fused Gram with one NCCL all-reduce (SURVEY.md section 8b / 8e) ----------------
 * Samples are independent: every device of the group runs the fused regressor -> normal-equation kernel on its own DEVICE-resident shard
 * and the only exchange is ONE ncclAllReduce(ncclDouble, ncclSum) of the packed partials [gram | rhs | tau_sq] (P^2 + P + 1 doubles) on
 * each device's stream -- no host round trip.  NCCL is bound at run time (dlopen "libnccl.so.2"; RDB_ERR_NOT_FOUND when a group of more than
 * one rank is asked for and it is absent).  Two ways to form a group:
 *   rdb_group_create      one process drives `ndev` devices (ncclCommInitAll); dev_ids NULL = devices 0 .. ndev-1.  This is what a C++
 *                         consumer such as rosdyn_identification (reference README.md:15) links against;
 *   rdb_group_create_rank one process per GPU (MPI / torchrun style, ncclCommInitRank): rank 0 calls rdb_group_unique_id and hands the 128
 *                         bytes to every rank out of band; the group then has ONE local device.
 * The group owns one chain handle per local device (rdb_group_chain: same chain, usable with every other entry point on that device).
 * rdb_regressor_gram_sharded: shards[k], tau_meas[k] (array or its entries may be NULL), gram[k] / rhs[k] / tau_sq[k] (entries may be NULL:
 * that device does not receive the result) are DEVICE pointers on local device k; streams[k] is the cudaStream_t of device k (an entry of 0 is
 * the default stream, as everywhere in CUDA); streams == NULL runs every device on the group's own stream (wait with rdb_group_synchronize).  Every non-NULL output receives the sum over ALL ranks (added to its contents when
 * accumulate != 0).  Asynchronous.  NCCL's summation order is fixed for a given number of ranks but differs from the single-GPU order:
 * compare with a tolerance, not bit for bit. */
typedef struct rdb_group rdb_group; /* opaque */
rdb_status rdb_group_create(const rdb_chain_desc* desc, int32_t ndev, const int32_t* dev_ids, rdb_group** out);
rdb_status rdb_group_unique_id(uint8_t id[128]);
rdb_status rdb_group_create_rank(const rdb_chain_desc* desc, int32_t device, int32_t nranks, int32_t rank, const uint8_t id[128],
                                 rdb_group** out);
void rdb_group_destroy(rdb_group* group);
int32_t rdb_group_size(const rdb_group* group);  /* local devices */
int32_t rdb_group_ranks(const rdb_group* group); /* ranks of the communicator */
rdb_chain* rdb_group_chain(rdb_group* group, int32_t k);
rdb_status rdb_regressor_gram_sharded(rdb_group* group, const rdb_samples* shards, const double* const* tau_meas, double* const* gram,
                                      double* const* rhs, double* const* tau_sq, int32_t accumulate, void* const* streams);
rdb_status rdb_group_synchronize(rdb_group* group);

/* ---- host-buffer convenience wrappers (pointers are HOST pointers; copies + sync inside) ----------
 * The handle is NOT const here: the staging buffers, streams and events of these pipelines live in the handle (grown on demand, freed with
 * it).  Calls on one handle from several host threads are serialised by a per-handle lock (they do not race, they do not overlap either);
 * for concurrency use one handle per thread, as the reference does with Chain::clone() (P.h:554).  Pinned (cudaHostAlloc /
 * cudaHostRegister) buffers overlap the copies with the kernels at the link's rate; pageable buffers work: the entries gather / scatter them
 * through pinned bounce buffers of the handle with a few host threads (0.5 - 0.6 of the link's rate; the driver's own staging reaches 0.2 - 0.3).
 * Calls whose arrays fit 256 KB in all (a handful of samples) skip the copies: the handle packs them into a mapped pinned buffer of its own
 * and the kernels work on it in place -- one launch and one synchronisation, 16-28 us per call on a B200 host (profiles/r02_latency.txt). */
rdb_status rdb_kinematics_batch_host(rdb_chain* chain, const rdb_samples* in, const rdb_kinematics_out* out);
rdb_status rdb_torque_batch_host(rdb_chain* chain, const rdb_samples* in, double* torque, int64_t ld_out);
rdb_status rdb_regressor_batch_host(rdb_chain* chain, const rdb_samples* in, double* phi, double* torque, int64_t ld_out);
rdb_status rdb_inertia_batch_host(rdb_chain* chain, const rdb_samples* in, double* inertia, int64_t ld_out);
rdb_status rdb_dynamics_batch_host(rdb_chain* chain, const rdb_samples* in, const rdb_dynamics_out* out);
rdb_status rdb_forward_dynamics_batch_host(rdb_chain* chain, const rdb_samples* in, const double* tau, double* ddq, int64_t ld_out,
                                           int32_t* info);
rdb_status rdb_regressor_gram_batch_host(rdb_chain* chain, const rdb_samples* in, const double* tau_meas, double* gram, double* rhs,
                                         double* tau_sq, int32_t accumulate);

/* ---- synthetic inputs (bench / tests): U(-1,1) from splitmix64, identical on host and device ------ */
/* x[plane][i] = 2 * (splitmix64(seed + 256*i + 64*stream_id + plane) >> 11) * 2^-53 - 1   (stream_id 0..3 = q, Dq, DDq, DDDq; plane < 64;
 * all sums modulo 2^64), with  splitmix64(x): x += 0x9E3779B97F4A7C15; x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9;
 * x = (x ^ (x >> 27)) * 0x94D049BB133111EB; return x ^ (x >> 31).  A reference-side harness that follows this formula gets bit-identical inputs
 * (tests/test_abi.py checks the documented formula against rdb_fill_uniform_host). */
rdb_status rdb_fill_uniform(double* x, int32_t n_planes, int64_t n, int64_t ld, uint64_t seed, int32_t stream_id, void* stream);
void rdb_fill_uniform_host(double* x, int32_t n_planes, int64_t n, int64_t ld, uint64_t seed, int32_t stream_id);

/* FP64 pipe micro-benchmarks (own roofline denominator; MEASURED_PEAKS.json carries no FP64 figure).
 * kind 0 = DFMA, 1 = DMMA m8n8k4, 2 = both interleaved (flops summed).  Returns achieved TFLOP/s in *tflops (CUDA-event timed, best of reps). */
rdb_status rdb_fp64_peak(int32_t kind, int32_t reps, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* ROSDYN_B200_H */
