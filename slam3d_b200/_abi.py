"""ctypes mirror of include/s3d_b200.h (struct layouts and status codes only; no logic)."""
import ctypes as C

S3D_OK = 0
S3D_TOO_FEW_POINTS = 1
S3D_NOT_CONVERGED = 2
S3D_TOO_FAR_FROM_GUESS = 3
S3D_UNKNOWN_ALGORITHM = 4
S3D_INTERNAL_ERROR = 5
S3D_INVALID_ARGUMENT = 6

ALG_ICP, ALG_GICP, ALG_GICP_OMP, ALG_NDT, ALG_NDT_OMP = range(5)

# s3d_set_gicp_optimizer: the inner optimiser of PCL's GICP (PCL >= 1.14 default / PCL <= 1.13)
GICP_NEWTON, GICP_BFGS = 0, 1
GICP_OPTIMIZERS = {"newton": GICP_NEWTON, "bfgs": GICP_BFGS}

# s3d_set_ndt_omp_search: the neighbour search of NDT_OMP (PCL's kd-tree radius search / pclomp's default DIRECT7)
NDT_OMP_KDTREE, NDT_OMP_DIRECT7 = 0, 1
NDT_OMP_SEARCHES = {"kdtree": NDT_OMP_KDTREE, "direct7": NDT_OMP_DIRECT7}


class RegistrationParameters(C.Structure):
    """slam3d::RegistrationParameters (RegistrationParameters.hpp:36-97), field for field."""
    _fields_ = [
        ("registration_algorithm", C.c_int32),
        ("point_cloud_density", C.c_double),
        ("max_fitness_score", C.c_double),
        ("max_translation", C.c_double),
        ("max_rotation", C.c_double),
        ("euclidean_fitness_epsilon", C.c_double),
        ("transformation_epsilon", C.c_double),
        ("max_correspondence_distance", C.c_double),
        ("maximum_iterations", C.c_int32),
        ("rotation_epsilon", C.c_double),
        ("correspondence_randomness", C.c_int32),
        ("maximum_optimizer_iterations", C.c_int32),
        ("resolution", C.c_float),
        ("step_size", C.c_double),
        ("outlier_ratio", C.c_double),
    ]

    @classmethod
    def defaults(cls, **kw):
        p = cls(ALG_GICP, 0.2, 2.0, 1.0, 1.0, 1.0, 1e-5, 2.5, 50, 2e-3, 20, 20, 1.0, 0.05, 0.35)
        for k, v in kw.items():
            if not hasattr(p, k):
                raise AttributeError(k)
            setattr(p, k, v)
        return p


class Cloud(C.Structure):
    _fields_ = [("xyzw", C.c_void_p), ("n", C.c_uint64)]


class Result(C.Structure):
    _fields_ = [
        ("T", C.c_double * 16),
        ("fitness", C.c_double),
        ("status", C.c_int32),
        ("converged", C.c_int32),
        ("outer_iterations", C.c_int32),
        ("inner_iterations", C.c_int32),
        ("n_source", C.c_uint32),
        ("n_target", C.c_uint32),
        ("n_correspondences", C.c_uint32),
        ("reserved", C.c_uint32),
    ]

    def pose(self):
        import numpy as np
        return np.array(self.T[:], dtype=np.float64).reshape(4, 4).T.copy()  # column-major -> [row, col]


class Counters(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]
