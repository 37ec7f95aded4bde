"""ctypes mirror of include/geoac_b200.h (POD types and enums only)."""
import ctypes as C

GEOAC_2D, GEOAC_3D, GEOAC_GLOBAL, GEOAC_3D_RNGDEP, GEOAC_GLOBAL_RNGDEP = range(5)
VARIANT_NAMES = {GEOAC_2D: "2d", GEOAC_3D: "3d", GEOAC_GLOBAL: "global",
                 GEOAC_3D_RNGDEP: "3drngdep", GEOAC_GLOBAL_RNGDEP: "globalrngdep"}

GEOAC_OK, GEOAC_ERR_NO_DEVICE, GEOAC_ERR_BAD_ARG, GEOAC_ERR_NO_ATMO, GEOAC_ERR_CUDA, GEOAC_ERR_TOO_LARGE, GEOAC_ERR_IO = range(7)

F_STATE0 = 0
F_TRAVELTIME, F_ATTEN, F_TURNHEIGHT, F_AMPLITUDE, F_INCLINATION, F_BACKAZ, F_AUX, F_MARGIN, F_JACOBIAN, F_CAUSTICS = range(18, 28)
NFIELDS = 28
CAUSTIC_NF = 6         # doubles per caustic event row: state[0..2], travel time, bounce, step
PATH_NF = 8            # doubles per raypath row (geoac_trace_paths): state[0..2], amplitude, absorption, travel time, bounce, step
ST_NONE, ST_ARRIVAL, ST_BREAK, ST_LIMIT = range(4)

# geoac_sample_atmosphere: rows of out[field][point]
ATM_C, ATM_U, ATM_V, ATM_RHO, ATM_DC, ATM_DU, ATM_DV, ATM_ALPHA = range(8)
ATM_T, ATM_UF, ATM_VF = 8, 18, 28     # each 10 rows: f, d0, d1, d2, d00, d11, d22, d01, d02, d12 over (p0, p1, p2)
ATM_NF = 38
SAMPLE_BLOCK = 1 << 20                # points per device pass


class GeoacParams(C.Structure):
    _fields_ = [
        ("ds_min", C.c_double), ("ds_max", C.c_double), ("ray_limit", C.c_double),
        ("vert_limit", C.c_double), ("range_limit", C.c_double),
        ("box_min", C.c_double * 2), ("box_max", C.c_double * 2),
        ("z_grnd", C.c_double), ("tweak_abs", C.c_double), ("freq", C.c_double),
        ("src", C.c_double * 3),
        ("bounces", C.c_int32), ("calc_amp", C.c_int32), ("accum_per_segment", C.c_int32), ("reserved", C.c_int32),
    ]

    def copy(self):
        q = GeoacParams()
        C.memmove(C.byref(q), C.byref(self), C.sizeof(self))
        return q


EIG_NF = 18            # doubles per eigenray-search row (geoac_eigenray_search)


class GeoacEigOpts(C.Structure):
    _fields_ = [
        ("theta_min", C.c_double), ("theta_max", C.c_double), ("azimuth_err_lim", C.c_double),
        ("d_theta_big", C.c_double), ("d_theta_small", C.c_double), ("tolerance", C.c_double),
        ("src_lat_deg", C.c_double), ("src_lon_deg", C.c_double),
        ("bnc_min", C.c_int32), ("bnc_max", C.c_int32), ("iterations", C.c_int32), ("max_rounds", C.c_int32),
    ]


def eq_count(variant, calc_amp):
    """GeoAc_SetEqCnt (reference Code/GeoAc/GeoAc.Interface.cpp:21-41)."""
    if variant == GEOAC_2D:
        return 6 if calc_amp else 3
    if variant == GEOAC_3D:
        return 12 if calc_amp else 4
    return 18 if calc_amp else 6
