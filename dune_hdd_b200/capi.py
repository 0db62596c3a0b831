"""ctypes binding of include/hdd_b200.h (libhdd_b200.so).

This is the raw C-ABI; the reference-shaped API lives in ``discretizations.py`` / ``estimators.py``.
The library is required: there is no CPU or torch fallback - a missing or unloadable extension raises.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

HDD_OK = 0
(HDD_ERR_WRONG_INPUT, HDD_ERR_USING_THIS_WRONG, HDD_ERR_WRONG_PARAMETER_TYPE, HDD_ERR_INDEX_OUT_OF_RANGE,
 HDD_ERR_NOT_IMPLEMENTED, HDD_ERR_REQUIREMENTS_NOT_MET, HDD_ERR_INTERNAL, HDD_ERR_DEVICE,
 HDD_ERR_NOT_CONVERGED) = range(1, 10)
HDD_SIMPLEX2D, HDD_CUBE2D = 0, 1
HDD_FN_CONSTANT, HDD_FN_CELLWISE, HDD_FN_EXPRESSION = 0, 1, 2
HDD_LHS, HDD_RHS = 0, 1


class hdd_function(C.Structure):
    _fields_ = [("kind", C.c_int), ("order", C.c_int), ("value", C.c_double),
                ("cell_values", C.POINTER(C.c_double)), ("expression", C.c_char_p)]


class hdd_affine_function(C.Structure):
    _fields_ = [("n_components", C.c_int), ("components", C.POINTER(hdd_function)),
                ("coefficients", C.POINTER(C.c_char_p)), ("affine_part", C.POINTER(hdd_function))]


class hdd_problem(C.Structure):
    _fields_ = [("diffusion_factor", hdd_affine_function), ("diffusion_tensor", C.POINTER(C.c_double)),
                ("force", hdd_affine_function), ("dirichlet", hdd_affine_function),
                ("neumann", hdd_affine_function), ("parameter_name", C.c_char_p), ("parameter_size", C.c_int)]


class hdd_solve_info(C.Structure):
    _fields_ = [("iterations", C.c_int), ("converged", C.c_int), ("relative_residual", C.c_double),
                ("seconds", C.c_double), ("seconds_per_iteration", C.c_double), ("peer_memory", C.c_int)]


class hdd_csr(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_cols", C.c_int64), ("nnz", C.c_int64), ("rowptr", C.POINTER(C.c_int64)),
                ("col", C.POINTER(C.c_int32)), ("val", C.POINTER(C.c_double))]


class hdd_parameters(C.Structure):
    _fields_ = [("mu", C.POINTER(C.c_double)), ("mu_hat", C.POINTER(C.c_double)), ("mu_bar", C.POINTER(C.c_double)),
                ("parameter_range_min", C.POINTER(C.c_double)), ("parameter_range_max", C.POINTER(C.c_double)),
                ("mu_size", C.c_int)]


# every symbol include/hdd_b200.h declares (checked by tests/test_host_logic.py)
SYMBOLS = [
    "hdd_last_error", "hdd_version", "hdd_mesh_create", "hdd_mesh_destroy", "hdd_mesh_num_cells",
    "hdd_grid_cube_sizes", "hdd_grid_cube", "hdd_grid_simplex_sizes", "hdd_grid_simplex", "hdd_swipdg_create",
    "hdd_swipdg_destroy", "hdd_swipdg_init", "hdd_swipdg_assemble", "hdd_num_dofs", "hdd_pattern",
    "hdd_num_components", "hdd_component_values", "hdd_component_coefficient", "hdd_evaluate_coefficients",
    "hdd_copy_to_host", "hdd_sync", "hdd_apply", "hdd_solver_types", "hdd_solve", "hdd_solution_dev",
    "hdd_num_subdomains", "hdd_subdomain_offsets", "hdd_neighbouring_subdomains", "hdd_block_extract",
    "hdd_csr_free", "hdd_estimators_available", "hdd_estimate", "hdd_indicators", "hdd_comm_unique_id",
    "hdd_comm_create", "hdd_comm_destroy", "hdd_mesh_attach_comm", "hdd_kernel_launches", "hdd_profile_kernel",
    "hdd_kernel_bytes", "hdd_expression_evaluate", "hdd_partition_plan", "hdd_free",
    "hdd_swipdg_only_these_products", "hdd_products_available", "hdd_product_num_components", "hdd_product_values",
    "hdd_product_coefficient", "hdd_pattern_volume", "hdd_product_apply2", "hdd_error_norms",
    "hdd_host_alloc", "hdd_host_free", "hdd_grid_fathers", "hdd_prolong", "hdd_residual", "hdd_partition_plan_local", "hdd_mesh_create_cube", "hdd_h2d_bytes",
]

# every symbol include/hdd_b200_testing.h declares: the entry points of the tests
TESTING_SYMBOLS = ["hdd_mg_strip_plan", "hdd_fast_cos", "hdd_trig_product", "hdd_precondition", "hdd_mg_level_operator"]

_lib = None


def library_path():
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libhdd_b200.so")


def lib():
    """Loads libhdd_b200.so (building it in-tree first if the sources are newer). Raises if it cannot."""
    global _lib
    if _lib is None:
        path = library_path()
        if os.path.exists(os.path.join(os.path.dirname(path), "csrc")) and os.path.exists(_build.NVCC):
            _build.build()
        if not os.path.exists(path):
            raise RuntimeError("libhdd_b200.so is missing; run `python -m dune_hdd_b200.build` (there is no fallback)")
        _lib = C.CDLL(path)
        _lib.hdd_last_error.restype = C.c_char_p
        _lib.hdd_version.restype = C.c_char_p
        _lib.hdd_kernel_launches.restype = C.c_int64
        _lib.hdd_h2d_bytes.restype = C.c_int64
    return _lib


class HddError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("[hdd status %d] %s" % (status, message))
        self.status = status
        self.message = message


def check(status):
    if status != HDD_OK:
        raise HddError(status, lib().hdd_last_error().decode())


def ptr(a, ctype=C.c_double):
    if a is None:
        return None
    return a.ctypes.data_as(C.POINTER(ctype))


def as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def as_i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


class _PinnedBlock:
    """page-locked host allocation (hdd_host_alloc) kept alive by the numpy arrays carved out of it"""

    def __init__(self, nbytes):
        self.ptr = C.c_void_p()
        self.nbytes = int(nbytes)
        check(lib().hdd_host_alloc(C.c_size_t(self.nbytes), C.byref(self.ptr)))

    def __del__(self):
        try:
            if self.ptr:
                lib().hdd_host_free(self.ptr)
        except Exception:
            pass


def pinned_empty(shape, dtype):
    """numpy array in page-locked host memory; falls back to ordinary memory if the allocation fails (no device)"""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape))
    try:
        blk = _PinnedBlock(max(n * dtype.itemsize, 1))
    except Exception:
        return np.empty(shape, dtype)
    buf = (C.c_char * blk.nbytes).from_address(blk.ptr.value)
    buf._hdd_owner = blk  # the ctypes buffer is the array's base object: the block lives as long as any view
    return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)


def h2d_bytes():
    return int(lib().hdd_h2d_bytes())


def kernel_launches():
    return int(lib().hdd_kernel_launches())
