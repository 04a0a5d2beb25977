"""ctypes binding of the C-ABI (include/rosdyn_b200.h).  Loads rosdyn_b200/librosdyn_b200.so and fails loudly
when it is missing: the product has no CPU / eager fallback."""
from __future__ import annotations

import ctypes
import os

from .descriptor import CChainDesc

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librosdyn_b200.so")  # the in-tree build, nothing else (no environment override)

_dp = ctypes.c_void_p  # device or host pointer to double
i32, i64, u64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64


class CSamples(ctypes.Structure):
    _fields_ = [("n", i64), ("ld", i64), ("q", _dp), ("dq", _dp), ("ddq", _dp), ("dddq", _dp)]


KIN_FIELDS = ("T_tool", "T_links", "jacobian", "twist", "dtwist", "dtwist_lin", "dtwist_nonlin", "ddtwist", "ddtwist_lin",
              "ddtwist_nonlin", "torque")


RDB_LAYOUT_SOA, RDB_LAYOUT_EIGEN = 0, 1


class CKinematicsOut(ctypes.Structure):
    _fields_ = [("ld", i64)] + [(k, _dp) for k in KIN_FIELDS] + [("layout", i32)]


class CDynamicsOut(ctypes.Structure):
    _fields_ = [("ld", i64), ("regressor", _dp), ("torque", _dp), ("inertia", _dp), ("layout", i32)]


class CUrdfChain(ctypes.Structure):
    _fields_ = [("desc", CChainDesc), ("joint_names", ctypes.POINTER(ctypes.c_char_p)), ("link_names", ctypes.POINTER(ctypes.c_char_p)),
                ("q_max", ctypes.POINTER(ctypes.c_double)), ("q_min", ctypes.POINTER(ctypes.c_double)), ("dq_max", ctypes.POINTER(ctypes.c_double)),
                ("ddq_max", ctypes.POINTER(ctypes.c_double)), ("tau_max", ctypes.POINTER(ctypes.c_double))]


class CComponentDesc(ctypes.Structure):
    _fields_ = [("type", i32), ("input_index", i32), ("min_velocity", ctypes.c_double), ("max_velocity", ctypes.c_double)]


# every symbol include/rosdyn_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "rdb_abi_version": (i32, []),
    "rdb_last_error": (ctypes.c_char_p, []),
    "rdb_status_string": (ctypes.c_char_p, [i32]),
    "rdb_device_count": (i32, []),
    "rdb_kernel_launch_count": (u64, []),
    "rdb_chain_create": (i32, [ctypes.POINTER(CChainDesc), ctypes.POINTER(ctypes.c_void_p)]),
    "rdb_chain_destroy": (None, [ctypes.c_void_p]),
    "rdb_chain_set_input_joints": (i32, [ctypes.c_void_p, i32, ctypes.POINTER(i32)]),
    "rdb_chain_joints_number": (i32, [ctypes.c_void_p]),
    "rdb_chain_links_number": (i32, [ctypes.c_void_p]),
    "rdb_chain_active_joints_number": (i32, [ctypes.c_void_p]),
    "rdb_chain_gravity": (i32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]),
    "rdb_chain_nominal_parameters": (i32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]),
    "rdb_urdf_parse": (i32, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.POINTER(CUrdfChain))]),
    "rdb_urdf_chain_free": (None, [ctypes.POINTER(CUrdfChain)]),
    "rdb_chain_from_urdf": (i32, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_void_p)]),
    "rdb_kinematics_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), ctypes.POINTER(CKinematicsOut), ctypes.c_void_p]),
    "rdb_torque_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, i64, ctypes.c_void_p]),
    "rdb_regressor_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, _dp, i64, ctypes.c_void_p]),
    "rdb_inertia_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, i64, ctypes.c_void_p]),
    "rdb_dynamics_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), ctypes.POINTER(CDynamicsOut), ctypes.c_void_p]),
    "rdb_dynamics_batch_host": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), ctypes.POINTER(CDynamicsOut)]),
    "rdb_forward_dynamics_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, _dp, i64, ctypes.c_void_p, ctypes.c_void_p]),
    "rdb_forward_dynamics_batch_host": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, _dp, i64, ctypes.c_void_p]),
    "rdb_regressor_gram_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, _dp, _dp, _dp, i32, ctypes.c_void_p]),
    "rdb_wrench_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, i64, _dp, _dp, i64, ctypes.c_void_p]),
    "rdb_jacobian_link_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), i32, _dp, i64, ctypes.c_void_p]),
    "rdb_local_ik_batch": (i32, [ctypes.c_void_p, i64, i64, _dp, _dp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                 ctypes.POINTER(ctypes.c_double), ctypes.c_double, i32, _dp, ctypes.c_void_p, ctypes.c_void_p, _dp,
                                 ctypes.c_void_p]),
    "rdb_component_columns": (i32, [i32]),
    "rdb_chain_set_components": (i32, [ctypes.c_void_p, i32, ctypes.POINTER(CComponentDesc)]),
    "rdb_chain_component_columns": (i32, [ctypes.c_void_p]),
    "rdb_components_regressor_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, i64, ctypes.c_void_p]),
    "rdb_components_torque_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), ctypes.POINTER(ctypes.c_double), _dp, i64, i32, ctypes.c_void_p]),
    "rdb_regressor_gram_ext_batch": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, _dp, _dp, _dp, i32, ctypes.c_void_p]),
    "rdb_fold_parameter_map": (i32, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    "rdb_fold_canonical_frame": (i32, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    "rdb_gram_row_layout": (i32, [i32, ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i32)]),
    "rdb_multiplicity": (i32, [i32, ctypes.POINTER(i32), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                               ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), i64, ctypes.POINTER(i64)]),
    "rdb_normal_equations_solve": (i32, [i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.c_double, ctypes.c_double,
                                         ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i32),
                                         ctypes.POINTER(ctypes.c_double)]),
    "rdb_kinematics_batch_host": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), ctypes.POINTER(CKinematicsOut)]),
    "rdb_torque_batch_host": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, i64]),
    "rdb_regressor_batch_host": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, _dp, i64]),
    "rdb_inertia_batch_host": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, i64]),
    "rdb_regressor_gram_batch_host": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), _dp, _dp, _dp, _dp, i32]),
    "rdb_chain_create_on": (i32, [ctypes.POINTER(CChainDesc), i32, ctypes.POINTER(ctypes.c_void_p)]),
    "rdb_chain_device": (i32, [ctypes.c_void_p]),
    "rdb_chain_gram_kernel_info": (i32, [ctypes.c_void_p, ctypes.POINTER(i32), ctypes.c_char_p, i32]),
    "rdb_gram_specialised_cubin": (i32, [ctypes.POINTER(CChainDesc), ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, i32]),
    "rdb_regressor_gram_sharded_host": (i32, [ctypes.POINTER(ctypes.c_void_p), i32, ctypes.POINTER(CSamples), _dp, _dp, _dp, _dp, i32]),
    "rdb_group_create": (i32, [ctypes.POINTER(CChainDesc), i32, ctypes.POINTER(i32), ctypes.POINTER(ctypes.c_void_p)]),
    "rdb_group_unique_id": (i32, [ctypes.POINTER(ctypes.c_uint8)]),
    "rdb_group_create_rank": (i32, [ctypes.POINTER(CChainDesc), i32, i32, i32, ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_void_p)]),
    "rdb_group_destroy": (None, [ctypes.c_void_p]),
    "rdb_group_size": (i32, [ctypes.c_void_p]),
    "rdb_group_ranks": (i32, [ctypes.c_void_p]),
    "rdb_group_chain": (ctypes.c_void_p, [ctypes.c_void_p, i32]),
    "rdb_regressor_gram_sharded": (i32, [ctypes.c_void_p, ctypes.POINTER(CSamples), ctypes.POINTER(_dp), ctypes.POINTER(_dp), ctypes.POINTER(_dp),
                                         ctypes.POINTER(_dp), i32, ctypes.POINTER(ctypes.c_void_p)]),
    "rdb_group_synchronize": (i32, [ctypes.c_void_p]),
    "rdb_fill_uniform": (i32, [_dp, i32, i64, i64, u64, i32, ctypes.c_void_p]),
    "rdb_fill_uniform_host": (None, [_dp, i32, i64, i64, u64, i32]),
    "rdb_fp64_peak": (i32, [i32, i32, ctypes.POINTER(ctypes.c_double)]),
}

RDB_OK, RDB_ERR_INVALID_ARG, RDB_ERR_DIM_MISMATCH, RDB_ERR_CUDA, RDB_ERR_NO_DEVICE, RDB_ERR_NOT_FOUND, RDB_ERR_ALLOC = range(7)

_lib = None


class RosdynB200Error(RuntimeError):
    def __init__(self, status: int, text: str):
        super().__init__(f"rosdyn_b200 status {status}: {text}")
        self.status = status


def set_library_path(path: str) -> None:
    """Development tools only (tools/bench_gram.py: A/B runs of experimental builds under build/var_*): must be called before the first load()."""
    global LIB_PATH
    if _lib is not None:
        raise RuntimeError("the library is already loaded")
    LIB_PATH = path


def load() -> ctypes.CDLL:
    """dlopen the in-tree C-ABI library and bind every declared symbol."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing - build it with `python -m rosdyn_b200.build` "
                              "(rosdyn_b200 has no CPU fallback)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status: int) -> None:
    if status == RDB_OK:
        return
    lib = load()
    msg = lib.rdb_last_error().decode() or lib.rdb_status_string(status).decode()
    if status == RDB_ERR_NOT_FOUND:
        # Chain ctor: throw std::runtime_error("Base link not found" / "Tool link not found") (primitives_impl.h:498-501, 601-613)
        raise LookupError(msg)
    if status == RDB_ERR_DIM_MISMATCH:
        # Chain::getRegressor throws std::invalid_argument("Input data dimensions mismatch") (primitives_impl.h:1299-1309)
        raise ValueError(msg)
    raise RosdynB200Error(status, msg)
