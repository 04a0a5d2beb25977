"""Host-side mirror of `rosdyn::Chain` over the C-ABI (reference: rosdyn_core/include/rosdyn_core/primitives.h:235-555).

Same method names and argument meaning as the reference; every method is ALSO its batched sibling:

* 1-D joint vectors (length n_act)          -> one sample, results shaped like the reference's Eigen objects;
* 2-D SoA arrays ``x[joint][N]`` (fp64)     -> N samples, results carry a trailing sample axis.

torch CUDA tensors go through the device entry points on torch's current stream (asynchronous, results are
torch CUDA tensors); numpy arrays go through the ``*_host`` entry points (copies + sync inside, results numpy).
torch is used for device memory and streams only.  There is no CPU fallback: constructing a Chain without the
built library or without a CUDA device raises.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import CKinematicsOut, CSamples, KIN_FIELDS, check
from .descriptor import ChainDesc, to_ctypes

try:  # torch is plumbing (device buffers, streams); the host (numpy) path works without it
    import torch
except Exception:  # pragma: no cover
    torch = None


def _ndim(x) -> int:
    return x.ndim if hasattr(x, "ndim") else np.ndim(x)


def _shape(x):
    return x.shape if hasattr(x, "shape") else np.shape(x)


def _is_torch(x) -> bool:
    return torch is not None and isinstance(x, torch.Tensor)


class Chain:
    """Batched B200 drop-in for rosdyn::Chain (hot path only: kinematics, twists, RNEA, regressor, inertia)."""

    def __init__(self, desc: ChainDesc, device: Optional[int] = None):
        """device: CUDA device index of the handle (None = the current device, as rdb_chain_create)."""
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        self.desc = desc
        cdesc, keep = to_ctypes(desc)
        if device is None:
            check(self._lib.rdb_chain_create(ctypes.byref(cdesc), ctypes.byref(self._h)))
        else:
            check(self._lib.rdb_chain_create_on(ctypes.byref(cdesc), int(device), ctypes.byref(self._h)))
        del keep
        self.nJ = self._lib.rdb_chain_joints_number(self._h)
        self.nL = self._lib.rdb_chain_links_number(self._h)
        self.n_in = self._lib.rdb_chain_active_joints_number(self._h)

    @classmethod
    def from_urdf(cls, urdf_xml: str, base_link: str, tool_link: str, gravity: Optional[Sequence[float]] = None) -> "Chain":
        """Chain(robot_description, base_link_name, ee_link_name, gravity) of the reference (primitives.h:349-352), with the
        library's own URDF loader; raises LookupError("Base link not found" / "Tool link not found")."""
        from .urdf import chain_from_urdf
        return cls(chain_from_urdf(urdf_xml, base_link, tool_link, gravity))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.rdb_chain_destroy(h)
            self._h = None

    # ------------------------------------------------------------------ metadata (primitives.h:364-447)
    def getJointsNumber(self) -> int:
        return self.nJ

    def getLinksNumber(self) -> int:
        return self.nL

    def getActiveJointsNumber(self) -> int:
        return self.n_in

    def getLinksName(self):
        return [l.name for l in self.desc.links]

    def getMoveableJointNames(self):
        return [j.name for j in self.desc.joints if j.type != 0]

    def getActiveJointsName(self):
        names = [None] * self.n_in
        for j in self.desc.joints:
            if j.input_index >= 0:
                names[j.input_index] = j.name
        return names

    def getGravity(self) -> np.ndarray:
        g = (ctypes.c_double * 3)()
        check(self._lib.rdb_chain_gravity(self._h, g))
        return np.array(g[:])

    def setInputJointsName(self, names: Sequence[str]) -> bool:
        """Chain::setInputJointsName (primitives_impl.h:705-742); False when a name is not in the chain."""
        idx = {j.name: k for k, j in enumerate(self.desc.joints)}
        sel = (ctypes.c_int32 * max(len(names), 1))(*[idx.get(n, -1) for n in names])
        check(self._lib.rdb_chain_set_input_joints(self._h, len(names), sel))
        ok = self.desc.set_input_joints(names)
        self.n_in = len(names)   # note: the C-ABI drops the additive components here (set them again with setComponents)
        return ok

    def getNominalParameters(self) -> np.ndarray:
        out = (ctypes.c_double * (10 * self.nJ))()
        check(self._lib.rdb_chain_nominal_parameters(self._h, out))
        return np.array(out[:])

    # ------------------------------------------------------------------ marshalling
    def _prep(self, arrays):
        """Returns (device?, single?, n, list of 2-D arrays or None)."""
        first = next(a for a in arrays if a is not None)
        dev = _is_torch(first) and first.is_cuda
        single = _ndim(first) == 1
        outs = []
        n = None
        for a in arrays:
            if a is None:
                outs.append(None)
                continue
            if _is_torch(a):
                if a.is_cuda != dev:
                    raise ValueError("all inputs must live on the same side (torch CUDA or host)")
                a = a.to(torch.float64)
                if a.ndim == 1:
                    a = a.reshape(-1, 1)
                if a.stride(-1) != 1:
                    a = a.contiguous()
                if not dev:
                    a = a.numpy()
            else:
                a = np.asarray(a, dtype=np.float64)
                if a.ndim == 1:
                    a = a.reshape(-1, 1)
                if a.strides[-1] != 8:
                    a = np.ascontiguousarray(a)
            if a.ndim != 2 or a.shape[0] != self.n_in:
                # the reference only checks sizes in getRegressor (primitives_impl.h:1299-1309); here every getter does
                raise ValueError("Input data dimensions mismatch")
            if n is None:
                n = a.shape[1]
            elif a.shape[1] != n:
                raise ValueError("Input data dimensions mismatch")
            outs.append(a)
        lds = {(_ld(a)) for a in outs if a is not None}
        if len(lds) > 1:  # the ABI takes one plane stride for all joint arrays
            outs = [None if a is None else (a.contiguous() if _is_torch(a) else np.ascontiguousarray(a)) for a in outs]
        return dev, single, n, outs

    def _with_tau(self, dev, n, arrs, tau_meas):
        """Measured torques for the normal equations: same side, same n_act x N shape as q (ValueError otherwise -- a shorter array would be
        read past its end), and brought to the one plane stride the ABI takes for q / Dq / DDq / tau_meas."""
        tdev, _, nt, (tau_arr,) = self._prep([tau_meas])
        if tdev != dev:
            raise ValueError("all inputs must live on the same side (torch CUDA or host)")
        if nt != n:
            raise ValueError("Input data dimensions mismatch")
        if _ld(tau_arr) != _ld(arrs[0]):
            tau_arr = tau_arr.contiguous() if _is_torch(tau_arr) else np.ascontiguousarray(tau_arr)
            if _ld(tau_arr) != _ld(arrs[0]):
                arrs = [None if a is None else (a.contiguous() if _is_torch(a) else np.ascontiguousarray(a)) for a in arrs]
        return arrs, tau_arr

    def _samples(self, n, arrs) -> CSamples:
        s = CSamples()
        s.n = n
        first = next(a for a in arrs if a is not None)
        s.ld = _ld(first)
        s.q, s.dq, s.ddq, s.dddq = (_ptr(a) for a in arrs)
        return s

    def _alloc(self, dev: bool, planes: int, n: int, like):
        if dev:
            return torch.empty((planes, n), dtype=torch.float64, device=like.device)
        return np.empty((planes, n), dtype=np.float64)

    @staticmethod
    def _stream():
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    # ------------------------------------------------------------------ kinematics
    def kinematics(self, q, Dq=None, DDq=None, DDDq=None, want: Sequence[str] = ("T_tool",), layout: str = "soa"):
        """One pass producing any subset of rdb_kinematics_out.  layout "soa": {name: planes[rows][N]} (raw plane layout);
        layout "eigen": {name: records[N][...]} shaped as the reference's Eigen containers lie in memory (RDB_LAYOUT_EIGEN):
        poses [N,4,4] views of the column-major Affine3d images (so r[i] reads as the 4x4 matrix), T_links [N,nL,4,4], 6-vectors [N,nL,6],
        jacobian [N,6,n_act], torque [N,n_act]."""
        dev, single, n, arrs = self._prep([q, Dq, DDq, DDDq])
        eig = {"soa": False, "eigen": True}[layout]
        pose = 16 if eig else 12
        rows = {"T_tool": pose, "T_links": pose * self.nL, "jacobian": 6 * self.n_in, "torque": self.n_in}
        out = CKinematicsOut()
        out.ld = max(n, 1)
        out.layout = _lib.RDB_LAYOUT_EIGEN if eig else _lib.RDB_LAYOUT_SOA
        res = {}
        for k in KIN_FIELDS:
            if k in want:
                r = rows.get(k, 6 * self.nL)
                res[k] = self._alloc(dev, n, r, arrs[0]) if eig else self._alloc(dev, r, n, arrs[0])
                setattr(out, k, _ptr(res[k]))
        s = self._samples(n, arrs)
        if dev:
            check(self._lib.rdb_kinematics_batch(self._h, ctypes.byref(s), ctypes.byref(out), self._stream()))
        else:
            check(self._lib.rdb_kinematics_batch_host(self._h, ctypes.byref(s), ctypes.byref(out)))
        if eig:  # shape the dense records like the Eigen objects (column-major matrices read through a transposed view)
            for k, r in res.items():
                if k == "T_tool":
                    res[k] = _swap_last2(r.reshape(n, 4, 4))
                elif k == "T_links":
                    res[k] = _swap_last2(r.reshape(n, self.nL, 4, 4))
                elif k == "jacobian":
                    res[k] = _swap_last2(r.reshape(n, self.n_in, 6))
                elif k != "torque":
                    res[k] = r.reshape(n, self.nL, 6)
        return res

    def dynamics(self, q, Dq=None, DDq=None, want: Sequence[str] = ("regressor", "torque"), layout: str = "soa"):
        """rdb_dynamics_batch: any subset of regressor / torque / inertia with a selectable layout.  "soa": raw planes
        {regressor [10 nJ * n_act][N], torque [n_act][N], inertia [n_act^2][N]}; "eigen": per-sample records viewed as the Eigen matrices
        {regressor [N, n_act, 10 nJ], torque [N, n_act], inertia [N, n_act, n_act]} (each record is the column-major matrix)."""
        if "regressor" in want and (Dq is None or DDq is None):
            raise ValueError("Input data dimensions mismatch")
        dev, single, n, arrs = self._prep([q, Dq, DDq, None])
        eig = {"soa": False, "eigen": True}[layout]
        P = 10 * self.nJ
        rows = {"regressor": P * self.n_in, "torque": self.n_in, "inertia": self.n_in * self.n_in}
        out = _lib.CDynamicsOut()
        out.ld = max(n, 1)
        out.layout = _lib.RDB_LAYOUT_EIGEN if eig else _lib.RDB_LAYOUT_SOA
        res = {}
        for k in ("regressor", "torque", "inertia"):
            if k in want:
                res[k] = self._alloc(dev, n, rows[k], arrs[0]) if eig else self._alloc(dev, rows[k], n, arrs[0])
                setattr(out, k, _ptr(res[k]))
        s = self._samples(n, arrs)
        if dev:
            check(self._lib.rdb_dynamics_batch(self._h, ctypes.byref(s), ctypes.byref(out), self._stream()))
        else:
            check(self._lib.rdb_dynamics_batch_host(self._h, ctypes.byref(s), ctypes.byref(out)))
        if eig:
            if "regressor" in res:
                res["regressor"] = _swap_last2(res["regressor"].reshape(n, P, self.n_in))
            if "inertia" in res:
                res["inertia"] = _swap_last2(res["inertia"].reshape(n, self.n_in, self.n_in))
        return res

    def _kin1(self, name, shape, q, Dq=None, DDq=None, DDDq=None):
        single = (_ndim(q) == 1)
        r = self.kinematics(q, Dq, DDq, DDDq, want=(name,))[name]
        r = r.reshape(*shape, r.shape[-1])
        return r[..., 0] if single else r

    def getTransformation(self, q):
        """Chain::getTransformation (PI.h:884): T_bt as 3x4 [R|p] (x N); a single sample returns the 4x4 Affine3d image."""
        r = self._kin1("T_tool", (3, 4), q)
        return _affine(r) if _ndim(q) == 1 else r

    computeTransformations = getTransformation  # name used by BASELINE.json's north_star (no such reference symbol)

    def getTransformations(self, q):
        """Chain::getTransformations (PI.h:908): all links, [nL,3,4(,N)]."""
        return self._kin1("T_links", (self.nL, 3, 4), q)

    def getJacobian(self, q):
        """Chain::getJacobian (PI.h:927): 6 x n_act (x N)."""
        r = self._kin1("jacobian", (self.n_in, 6), q)
        return _swap01(r)

    def getTwist(self, q, Dq):
        return self._kin1("twist", (self.nL, 6), q, Dq)

    def getTwistTool(self, q, Dq):
        return self.getTwist(q, Dq)[-1]

    def getDTwist(self, q, Dq, DDq):
        return self._kin1("dtwist", (self.nL, 6), q, Dq, DDq)

    def getDTwistTool(self, q, Dq, DDq):
        return self.getDTwist(q, Dq, DDq)[-1]

    def getDTwistLinearPart(self, q, DDq):
        return self._kin1("dtwist_lin", (self.nL, 6), q, None, DDq)

    def getDTwistNonLinearPart(self, q, Dq):
        return self._kin1("dtwist_nonlin", (self.nL, 6), q, Dq)

    def getDDTwist(self, q, Dq, DDq, DDDq):
        return self._kin1("ddtwist", (self.nL, 6), q, Dq, DDq, DDDq)

    def getDDTwistTool(self, q, Dq, DDq, DDDq):
        return self.getDDTwist(q, Dq, DDq, DDDq)[-1]

    def getDDTwistLinearPart(self, q, DDDq):
        return self._kin1("ddtwist_lin", (self.nL, 6), q, None, None, DDDq)

    def getDDTwistNonLinearPart(self, q, Dq, DDq):
        return self._kin1("ddtwist_nonlin", (self.nL, 6), q, Dq, DDq)

    # ------------------------------------------------------------------ dynamics
    def getJointTorque(self, q, Dq, DDq):
        """Chain::getJointTorque(q,Dq,DDq) (PI.h:1277): n_act (x N)."""
        dev, single, n, arrs = self._prep([q, Dq, DDq, None])
        tau = self._alloc(dev, self.n_in, n, arrs[0])
        s = self._samples(n, arrs)
        if dev:
            check(self._lib.rdb_torque_batch(self._h, ctypes.byref(s), _ptr(tau), max(n, 1), self._stream()))
        else:
            check(self._lib.rdb_torque_batch_host(self._h, ctypes.byref(s), _ptr(tau), max(n, 1)))
        return tau[:, 0] if single else tau

    def getWrench(self, q, Dq, DDq, ext_wrenches_in_link_frame=None, with_torque: bool = False):
        """Chain::getWrench (PI.h:1225-1262): nL x 6 (x N), base frame at each link origin; external wrenches nL x 6 (x N) are applied
        TO the links in link frames.  with_torque also returns getJointTorque(q,Dq,DDq,ext) (PI.h:1264-1274).  Device arrays only."""
        dev, single, n, arrs = self._prep([q, Dq, DDq, None])
        if not dev:
            raise ValueError("getWrench takes device (torch CUDA) arrays")
        ext = None
        if ext_wrenches_in_link_frame is not None:
            ext = ext_wrenches_in_link_frame.to(torch.float64).reshape(6 * self.nL, -1).contiguous()
            if ext.shape[1] != n:
                raise ValueError("Input data dimensions mismatch")
        w = self._alloc(dev, 6 * self.nL, n, arrs[0])
        tau = self._alloc(dev, self.n_in, n, arrs[0]) if with_torque else None
        s = self._samples(n, arrs)
        check(self._lib.rdb_wrench_batch(self._h, ctypes.byref(s), _ptr(ext), max(n, 1), _ptr(tau), _ptr(w), max(n, 1), self._stream()))
        w = w.reshape(self.nL, 6, n)
        if single:
            w = w[..., 0]
            tau = tau[:, 0] if tau is not None else None
        return (w, tau) if with_torque else w

    def getJacobianLink(self, q, link_name):
        """Chain::getJacobianLink(q, link_name) (PI.h:951-979): 6 x n_act (x N); std::invalid_argument for a link outside the chain."""
        names = self.getLinksName()
        if isinstance(link_name, str):
            if link_name not in names:
                raise ValueError(f"link {link_name} is not member of the chain")
            link_name = names.index(link_name)
        dev, single, n, arrs = self._prep([q, None, None, None])
        if not dev:
            raise ValueError("getJacobianLink takes device (torch CUDA) arrays")
        J = self._alloc(dev, 6 * self.n_in, n, arrs[0])
        s = self._samples(n, arrs)
        check(self._lib.rdb_jacobian_link_batch(self._h, ctypes.byref(s), int(link_name), _ptr(J), max(n, 1), self._stream()))
        r = _swap01(J.reshape(self.n_in, 6, n))
        return r[..., 0] if single else r

    def computeLocalIk(self, T_b_t, seed, q_min=None, q_max=None, weight=None, toll: float = 1e-6, max_iter: int = 50):
        """Chain::computeLocalIk / computeWeigthedLocalIk (PI.h:1398-1468), batched over N target poses.
        T_b_t: 12 planes (3x4 [R|p] row-major, as kinematics(...)["T_tool"] returns them) x N, or one 4x4 / 3x4 pose; seed: n_act (x N).
        The reference's wall-clock budget is an iteration budget (max_iter).  Returns (sol, converged, iterations, error_norm).
        Device (torch CUDA) arrays only; q_min / q_max / weight are small host arrays (None = no limits / unweighted)."""
        if not _is_torch(T_b_t) or not T_b_t.is_cuda:
            raise ValueError("computeLocalIk takes device (torch CUDA) arrays")
        single = seed.dim() == 1
        T = T_b_t.to(torch.float64)
        if single:
            T = T[:3, :].reshape(12, 1)
        T = T.reshape(12, -1).contiguous()
        sd = seed.to(torch.float64).reshape(self.n_in, -1).contiguous()
        n = T.shape[1]
        if sd.shape[1] != n:
            raise ValueError("Input data dimensions mismatch")

        def host(a, m):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.float64)
            if a.shape != (m,):
                raise ValueError("Input data dimensions mismatch")
            return a
        qmin, qmax, w = host(q_min, self.n_in), host(q_max, self.n_in), host(weight, 6)
        dp = ctypes.POINTER(ctypes.c_double)
        hp = lambda a: None if a is None else a.ctypes.data_as(dp)  # noqa: E731
        sol = torch.empty((self.n_in, max(n, 1)), dtype=torch.float64, device=T.device)[:, :n]
        stat = torch.zeros((max(n, 1),), dtype=torch.int32, device=T.device)[:n]
        its = torch.zeros((max(n, 1),), dtype=torch.int32, device=T.device)[:n]
        err = torch.zeros((max(n, 1),), dtype=torch.float64, device=T.device)[:n]
        check(self._lib.rdb_local_ik_batch(self._h, n, max(n, 1), _ptr(T), _ptr(sd), hp(qmin), hp(qmax), hp(w), float(toll), int(max_iter),
                                           _ptr(sol), _ptr(stat), _ptr(its), _ptr(err), self._stream()))
        if single:
            return sol[:, 0], bool(stat[0].item()), int(its[0].item()), float(err[0].item())
        return sol, stat, its, err

    computeWeigthedLocalIk = computeLocalIk  # the reference's spelling (PI.h:1435); pass weight=

    def getMultiplicity(self, q, q_min, q_max):
        """Chain::getMultiplicity (PI.h:1470-1517): the multi-turn images q + 2 pi k of a joint vector inside the limits (revolute input joints
        only), in the reference's order; host arrays.  Returns an array [count][n_act]."""
        return multiplicity(self._input_joint_types(), q, q_min, q_max)

    def _input_joint_types(self):
        t = [0] * self.n_in
        for j in self.desc.joints:
            if 0 <= j.input_index < self.n_in:
                t[j.input_index] = int(j.type)
        return t

    def getTransformationLink(self, q, link_name):
        """Chain::getTransformationLink (PI.h:912-925)."""
        names = self.getLinksName()
        if link_name not in names:
            raise ValueError(f"link {link_name} is not member of the chain")
        return self.getTransformations(q)[names.index(link_name)]

    def getTwistLink(self, q, Dq, link_name):
        """Chain::getTwistLink (PI.h:1016-1027)."""
        names = self.getLinksName()
        if link_name not in names:
            raise ValueError(f"link {link_name} is not member of the chain")
        return self.getTwist(q, Dq)[names.index(link_name)]

    def getJointTorqueNonLinearPart(self, q, Dq):
        """PI.h:1285-1293: getJointTorque with DDq = 0."""
        return self.getJointTorque(q, Dq, None)

    def getRegressor(self, q, Dq, DDq, with_torque: bool = False):
        """Chain::getRegressor (PI.h:1295): n_act x 10*nJ (x N).  with_torque also returns getJointTorque of the
        same samples from the same pass."""
        if Dq is None or DDq is None or tuple(_shape(q)) != tuple(_shape(Dq)) or tuple(_shape(Dq)) != tuple(_shape(DDq)):
            raise ValueError("Input data dimensions mismatch")
        dev, single, n, arrs = self._prep([q, Dq, DDq, None])
        P = 10 * self.nJ
        phi = self._alloc(dev, P * self.n_in, n, arrs[0])
        tau = self._alloc(dev, self.n_in, n, arrs[0]) if with_torque else None
        s = self._samples(n, arrs)
        if dev:
            check(self._lib.rdb_regressor_batch(self._h, ctypes.byref(s), _ptr(phi), _ptr(tau), max(n, 1), self._stream()))
        else:
            check(self._lib.rdb_regressor_batch_host(self._h, ctypes.byref(s), _ptr(phi), _ptr(tau), max(n, 1)))
        r = _swap01(phi.reshape(P, self.n_in, n))
        if single:
            r = r[..., 0]
            tau = tau[:, 0] if tau is not None else None
        return (r, tau) if with_torque else r

    def getJointInertia(self, q):
        """Chain::getJointInertia (PI.h:1357): n_act x n_act (x N)."""
        dev, single, n, arrs = self._prep([q, None, None, None])
        M = self._alloc(dev, self.n_in * self.n_in, n, arrs[0])
        s = self._samples(n, arrs)
        if dev:
            check(self._lib.rdb_inertia_batch(self._h, ctypes.byref(s), _ptr(M), max(n, 1), self._stream()))
        else:
            check(self._lib.rdb_inertia_batch_host(self._h, ctypes.byref(s), _ptr(M), max(n, 1)))
        r = _swap01(M.reshape(self.n_in, self.n_in, n))
        return r[..., 0] if single else r

    def getJointAcceleration(self, q, Dq, tau, with_info: bool = False):
        """Forward dynamics ddq = M(q)^-1 (tau - h(q, Dq)) with h = getJointTorque(q, Dq, 0) (rdb_forward_dynamics_batch): n_act (x N).
        Dq / tau may be None (zero).  with_info also returns info, int32 (N,) (or an int for 1-D inputs): 1 where M(q) is not positive
        definite (that sample's ddq is all NaN), else 0.  Torch CUDA arrays run on the device, host arrays through the host twin."""
        dev, single, n, arrs = self._prep([q, Dq, None, None])
        tau_arr = None
        if tau is not None:
            arrs, tau_arr = self._with_tau(dev, n, arrs, tau)
        ddq = self._alloc(dev, self.n_in, n, arrs[0])
        info = None
        if with_info:
            info = torch.empty((max(n, 1),), dtype=torch.int32, device=arrs[0].device)[:n] if dev else np.empty((n,), dtype=np.int32)
        s = self._samples(n, arrs)
        if dev:
            check(self._lib.rdb_forward_dynamics_batch(self._h, ctypes.byref(s), _ptr(tau_arr), _ptr(ddq), max(n, 1), _ptr(info), self._stream()))
        else:
            check(self._lib.rdb_forward_dynamics_batch_host(self._h, ctypes.byref(s), _ptr(tau_arr), _ptr(ddq), max(n, 1), _ptr(info)))
        if single:
            ddq = ddq[:, 0]
            info = int(info[0]) if info is not None else None
        return (ddq, info) if with_info else ddq

    def gramKernelInfo(self):
        """(specialised, reason) of the kernel the last regressorGram* call ran: 1 fused kernel compiled at run time against this chain's
        constants, 0 precompiled fused kernel, 2 general pipeline (more than 7 moving joints, no moving joint, or a component set the
        one-pass kernel refuses; reason starts with "general pipeline:"), -1 no call yet (rdb_chain_gram_kernel_info)."""
        flag = ctypes.c_int32(-1)
        buf = ctypes.create_string_buffer(4096)
        check(self._lib.rdb_chain_gram_kernel_info(self._h, ctypes.byref(flag), buf, len(buf)))
        return flag.value, buf.value.decode(errors="replace")

    def regressorGram(self, q, Dq, DDq, tau_meas=None, out=None):
        """Fused getRegressor -> normal equations: returns (G[P,P], b[P], tau_sq[1]) with
        G = sum Phi^T Phi, b = sum Phi^T tau, tau_sq = sum tau^T tau; tau = tau_meas or getJointTorque.
        `out=(G,b,tau_sq)` accumulates into existing arrays (chunked / multi-pass use)."""
        if Dq is None or DDq is None:
            raise ValueError("Input data dimensions mismatch")
        dev, single, n, arrs = self._prep([q, Dq, DDq, None])
        tau_arr = None
        if tau_meas is not None:
            arrs, tau_arr = self._with_tau(dev, n, arrs, tau_meas)
        P = 10 * self.nJ
        acc = out is not None
        if acc:
            G, b, tt = out
        elif dev:
            G = torch.empty((P, P), dtype=torch.float64, device=arrs[0].device)
            b = torch.empty((P,), dtype=torch.float64, device=arrs[0].device)
            tt = torch.empty((1,), dtype=torch.float64, device=arrs[0].device)
        else:
            G, b, tt = np.empty((P, P)), np.empty((P,)), np.empty((1,))
        s = self._samples(n, arrs)
        if dev:
            check(self._lib.rdb_regressor_gram_batch(self._h, ctypes.byref(s), _ptr(tau_arr), _ptr(G), _ptr(b), _ptr(tt), int(acc), self._stream()))
        else:
            check(self._lib.rdb_regressor_gram_batch_host(self._h, ctypes.byref(s), _ptr(tau_arr), _ptr(G), _ptr(b), _ptr(tt), int(acc)))
        return G, b, tt


    # ------------------------------------------------------------------ additive joint components (SURVEY.md 8f N2)
    def setComponents(self, components: Sequence[dict]) -> int:
        """components: [{"type": "friction1" | "friction2" | "spring", "joint": <input joint name or index>,
        "min_velocity": .., "max_velocity": ..}, ...] in column order (FirstOrderPolynomialFriction / SecondOrderPolynomialFriction /
        IdealSpring, friction_polynomial1.h, friction_polynomial2.h, ideal_spring.h).  Returns the number of component columns."""
        from ._lib import CComponentDesc
        types = {"friction1": 1, "friction2": 2, "spring": 3}
        names = self.getActiveJointsName()
        arr = (CComponentDesc * max(len(components), 1))()
        for k, c in enumerate(components):
            j = c["joint"]
            if isinstance(j, str):
                if j not in names:
                    # ComponentBase ctor: std::invalid_argument("Component Joint name ... is not a elemente of ...") (base_component.h:103)
                    raise LookupError(f"Component Joint name '{j}' is not an input joint")
                j = names.index(j)
            arr[k].type = types[c["type"]] if isinstance(c["type"], str) else int(c["type"])
            arr[k].input_index = int(j)
            arr[k].min_velocity = float(c.get("min_velocity", 0.0))
            arr[k].max_velocity = float(c.get("max_velocity", 0.0))
        check(self._lib.rdb_chain_set_components(self._h, len(components), arr))
        return self.getComponentColumns()

    def getComponentColumns(self) -> int:
        return int(self._lib.rdb_chain_component_columns(self._h))

    def getComponentsRegressor(self, q, Dq):
        """ComponentBase::getRegressor of every component side by side: n_act x Pc (x N); device arrays only."""
        dev, single, n, arrs = self._prep([q, Dq, None, None])
        if not dev:
            raise ValueError("component entry points take device (torch CUDA) arrays")
        Pc = self.getComponentColumns()
        phi = self._alloc(dev, Pc * self.n_in, n, arrs[0])
        s = self._samples(n, arrs)
        check(self._lib.rdb_components_regressor_batch(self._h, ctypes.byref(s), _ptr(phi), max(n, 1), self._stream()))
        r = _swap01(phi.reshape(Pc, self.n_in, n))
        return r[..., 0] if single else r

    def getComponentsTorque(self, q, Dq, parameters, out=None):
        """Sum of ComponentBase::getTorque over the components (regressor * parameters); `out` accumulates onto an existing torque."""
        dev, single, n, arrs = self._prep([q, Dq, None, None])
        if not dev:
            raise ValueError("component entry points take device (torch CUDA) arrays")
        prm = np.ascontiguousarray(parameters, dtype=np.float64)
        if prm.shape != (self.getComponentColumns(),):
            raise ValueError("Input data dimensions mismatch")
        tau = out if out is not None else self._alloc(dev, self.n_in, n, arrs[0])
        s = self._samples(n, arrs)
        check(self._lib.rdb_components_torque_batch(self._h, ctypes.byref(s), prm.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), _ptr(tau),
                                                    _ld(tau), int(out is not None), self._stream()))
        return tau[:, 0] if (single and out is None) else tau

    def regressorGramExt(self, q, Dq, DDq, tau_meas=None, out=None):
        """Normal equations of the extended model [Phi | Phi_components]: (G[Pt,Pt], b[Pt], tau_sq[1]), Pt = 10*nJ + Pc."""
        dev, single, n, arrs = self._prep([q, Dq, DDq, None])
        if not dev:
            raise ValueError("component entry points take device (torch CUDA) arrays")
        tau_arr = None
        if tau_meas is not None:
            arrs, tau_arr = self._with_tau(dev, n, arrs, tau_meas)
        Pt = 10 * self.nJ + self.getComponentColumns()
        acc = out is not None
        if acc:
            G, b, tt = out
        else:
            G = torch.empty((Pt, Pt), dtype=torch.float64, device=arrs[0].device)
            b = torch.empty((Pt,), dtype=torch.float64, device=arrs[0].device)
            tt = torch.empty((1,), dtype=torch.float64, device=arrs[0].device)
        s = self._samples(n, arrs)
        check(self._lib.rdb_regressor_gram_ext_batch(self._h, ctypes.byref(s), _ptr(tau_arr), _ptr(G), _ptr(b), _ptr(tt), int(acc), self._stream()))
        return G, b, tt


# ---------------------------------------------------------------------- helpers
def _ptr(a):
    if a is None:
        return None
    if _is_torch(a):
        return ctypes.c_void_p(a.data_ptr())
    return ctypes.c_void_p(a.ctypes.data)


def _ld(a) -> int:
    if _is_torch(a):
        return int(a.stride(0)) if a.shape[0] > 1 else max(int(a.shape[1]), 1)
    return int(a.strides[0] // 8) if a.shape[0] > 1 else max(int(a.shape[1]), 1)


def _swap01(a):
    return a.transpose(0, 1) if _is_torch(a) else np.swapaxes(a, 0, 1)


def _swap_last2(a):
    return a.transpose(-1, -2) if _is_torch(a) else np.swapaxes(a, -1, -2)


def _affine(r34):
    if _is_torch(r34):
        T = torch.eye(4, dtype=torch.float64, device=r34.device)
        T[:3, :] = r34
        return T
    T = np.eye(4)
    T[:3, :] = r34
    return T


def fill_uniform(n_planes: int, n: int, seed: int, stream_id: int, device=None):
    """U(-1,1) synthetic joint samples x[plane][n] (rdb_fill_uniform): torch CUDA tensor, or numpy when device is None."""
    lib = _lib.load()
    if device is None:
        x = np.empty((n_planes, n))
        lib.rdb_fill_uniform_host(_ptr(x), n_planes, n, max(n, 1), seed, stream_id)
        return x
    x = torch.empty((n_planes, n), dtype=torch.float64, device=device)
    check(lib.rdb_fill_uniform(_ptr(x), n_planes, n, max(n, 1), seed, stream_id, Chain._stream()))
    return x


def solveNormalEquations(G, b, tau_sq=0.0, rel_tol: float = 1e-10):
    """Minimum-norm least-squares solution of G pi = b (host, fp64; SURVEY.md 8f N3).  G, b: numpy or torch (copied to the host).
    Returns dict(parameters, eigenvalues, rank, residual_sq)."""
    lib = _lib.load()
    Gh = np.ascontiguousarray(G.detach().cpu().numpy() if _is_torch(G) else G, dtype=np.float64)
    bh = np.ascontiguousarray(b.detach().cpu().numpy() if _is_torch(b) else b, dtype=np.float64)
    tt = float(tau_sq.reshape(-1)[0]) if hasattr(tau_sq, "reshape") else float(tau_sq)
    P = bh.shape[0]
    if Gh.shape != (P, P):
        raise ValueError("Input data dimensions mismatch")
    prm, ev = np.zeros(P), np.zeros(P)
    rank, res = ctypes.c_int32(0), ctypes.c_double(0.0)
    dp = ctypes.POINTER(ctypes.c_double)
    check(lib.rdb_normal_equations_solve(P, Gh.ctypes.data_as(dp), bh.ctypes.data_as(dp), tt, float(rel_tol), prm.ctypes.data_as(dp),
                                         ev.ctypes.data_as(dp), ctypes.byref(rank), ctypes.byref(res)))
    return {"parameters": prm, "eigenvalues": ev, "rank": int(rank.value), "residual_sq": float(res.value)}


def fp64_peak(kind: str = "dmma", reps: int = 5) -> float:
    """Own FP64 roofline denominator in TFLOP/s: 'dfma' (vector pipe) or 'dmma' (mma.sync m8n8k4 f64)."""
    v = ctypes.c_double()
    check(_lib.load().rdb_fp64_peak({"dfma": 0, "dmma": 1, "mixed": 2}[kind], reps, ctypes.byref(v)))
    return float(v.value)


def kernel_launch_count() -> int:
    return int(_lib.load().rdb_kernel_launch_count())


def createChain(model, base_frame: Optional[str] = None, tool_frame: Optional[str] = None,
                gravity: Optional[Sequence[float]] = None) -> Optional[Chain]:
    """rosdyn::createChain(urdf_model, base_frame, tool_frame, gravity) (primitives_impl.h:1518-1527).  `model` is a URDF string
    (with base/tool frames) or a ChainDesc; like the reference it returns None instead of raising when the chain cannot be built."""
    try:
        if isinstance(model, str):
            return Chain.from_urdf(model, base_frame, tool_frame, gravity)
        if gravity is not None:
            model.gravity = tuple(gravity)
        return Chain(model)
    except (LookupError, ValueError):
        return None
    except _lib.RosdynB200Error as e:
        if e.status == _lib.RDB_ERR_INVALID_ARG:
            return None
        raise


def multiplicity(joint_type_of_input, q, q_min, q_max):
    """rdb_multiplicity (host only, no device needed): see Chain.getMultiplicity."""
    from ._lib import load
    lib = load()
    n = len(joint_type_of_input)
    ty = (ctypes.c_int32 * max(n, 1))(*[int(v) for v in joint_type_of_input])
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (q, q_min, q_max)]
    if any(a.shape != (n,) for a in arrs):
        raise ValueError("Input data dimensions mismatch")
    dp = ctypes.POINTER(ctypes.c_double)
    cnt = ctypes.c_int64(0)
    lib.rdb_multiplicity(n, ty, *[a.ctypes.data_as(dp) for a in arrs], None, 0, ctypes.byref(cnt))  # first call: how many
    out = np.zeros((cnt.value, n))
    check(lib.rdb_multiplicity(n, ty, *[a.ctypes.data_as(dp) for a in arrs], out.ctypes.data_as(dp), cnt.value, ctypes.byref(cnt)))
    return out
