"""ctypes mirrors of the kernel parameter structs (csrc/cuda/*.cu)."""
import ctypes as C

MAX_ROWS = 512
MAX_PEERS = 8
fptr = C.c_void_p


class Epilogue(C.Structure):
    _fields_ = [("out", fptr * MAX_PEERS), ("theta", fptr * MAX_PEERS), ("theta_src", fptr),
                ("lr", C.c_float), ("n_out", C.c_int), ("n_theta", C.c_int),
                ("mc_out", fptr), ("mc_theta", fptr)]         # NVLS multicast addresses (0: one store per peer)


class SelectParams(C.Structure):
    _fields_ = [("rows", fptr * 128), ("n_real", C.c_int), ("n_stat", C.c_int), ("n_virtual", C.c_int),
                ("virt_kind", C.c_int), ("virt_param", C.c_float), ("mode", C.c_int), ("trim_b", C.c_int),
                ("c0", C.c_longlong), ("c1", C.c_longlong), ("ep", Epilogue),
                ("virt_param_ptr", fptr)]     # device-resident virt_param (scale solver); 0: use virt_param


class SelectLargeParams(C.Structure):
    _fields_ = [("rows", fptr * MAX_ROWS), ("n_real", C.c_int), ("n_stat", C.c_int), ("n_virtual", C.c_int),
                ("virt_kind", C.c_int), ("virt_param", C.c_float), ("mode", C.c_int), ("trim_b", C.c_int),
                ("c0", C.c_longlong), ("c1", C.c_longlong), ("ep", Epilogue), ("virt_param_ptr", fptr)]


class CombineParams(C.Structure):
    _fields_ = [("rows", fptr * (MAX_ROWS + 1)), ("w", C.c_float * (MAX_ROWS + 1)), ("n_rows", C.c_int),
                ("c0", C.c_longlong), ("c1", C.c_longlong), ("ep", Epilogue), ("ep_vec", C.c_int),
                ("w_dev", fptr)]          # device-resident weights (on-device Gram solvers); overrides w


class AttackRowParams(C.Structure):
    _fields_ = [("rows", fptr * MAX_ROWS), ("n_stat", C.c_int), ("kind", C.c_int), ("param", C.c_float),
                ("c0", C.c_longlong), ("c1", C.c_longlong), ("out", fptr * MAX_ROWS), ("n_out", C.c_int),
                ("param_ptr", fptr)]


class DeviationParams(C.Structure):
    _fields_ = [("rows", fptr * MAX_ROWS), ("n_stat", C.c_int), ("dev_type", C.c_int),
                ("c0", C.c_longlong), ("c1", C.c_longlong), ("q", fptr)]


def verify(lib) -> None:
    for fn, st in (("bl_sizeof_select_params", SelectParams),
                   ("bl_sizeof_select_large_params", SelectLargeParams),
                   ("bl_sizeof_combine_params", CombineParams),
                   ("bl_sizeof_attack_params", AttackRowParams),
                ("bl_sizeof_deviation_params", DeviationParams)):
        got = getattr(lib, fn)()
        assert got == C.sizeof(st), f"{fn}: C={got} ctypes={C.sizeof(st)}"
