"""ctypes binding of liblbm_b200.so (include/lbm_b200.h) — plumbing only.

The product is the CUDA library; this module just loads it, mirrors the C structs and moves
numpy buffers across the C ABI.  It fails loudly when the library is missing: there is no CPU
or PyTorch fallback for any compute entry point.
"""
import ctypes as C
import os

import numpy as np

PKG_DIR = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
LIB_PATH = os.path.join(PKG_DIR, "liblbm_b200.so")

LBM_END = 2147483647

# enums of include/lbm_b200.h
MODEL_BGK, MODEL_BGK_ADE, MODEL_MRTCG, MODEL_RK, MODEL_KBC, MODEL_MRT_CSF = 0, 1, 2, 3, 4, 5
EQ_COMPRESSIBLE, EQ_INCOMPRESSIBLE, EQ_KBC, EQ_KBC_FRESH = 0, 1, 2, 3
FORCE_NONE, FORCE_UNIFORM, FORCE_IBM = 0, 1, 2
BC_LINEAR, BC_ABB_FIXED, BC_ABB_EXTRAPOLATED, BC_ADE_INLET, BC_PRESSURE_PERIODIC, BC_COPY_PRE = range(6)
SRC_SAME_NODE, SRC_SHIFT, SRC_ROW, SRC_COL = range(4)
OK, ERR_INVALID, ERR_CUDA, ERR_CONFIG, ERR_UNSUPPORTED, ERR_COMM = range(6)
UNIQUE_ID_BYTES = 128

OPP = [0, 3, 4, 1, 2, 7, 8, 5, 6]

dp = C.POINTER(C.c_double)


class LbmError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"lbm_b200 status {status}: {message}")
        self.status = status
        self.message = message


class ColourDesc(C.Structure):
    _fields_ = [("rho_0", C.c_double), ("alpha", C.c_double), ("A", C.c_double), ("nu", C.c_double), ("beta", C.c_double)]


class Config(C.Structure):
    _fields_ = [
        ("model", C.c_int), ("X", C.c_int), ("Y", C.c_int), ("x0", C.c_int), ("x1", C.c_int), ("device", C.c_int),
        ("omega", C.c_double), ("equilibrium", C.c_int), ("force", C.c_int), ("Fg", C.c_double * 2),
        ("w_s", C.c_double), ("omega_g", C.c_double),
        ("red", ColourDesc), ("blue", ColourDesc), ("sigma", C.c_double), ("delta", C.c_double), ("add_force", C.c_int),
    ]


class RkDiag(C.Structure):
    """lbm_rk_diag: host output pointers of lbm_rk_diagnostics"""
    FIELDS = (("phase", ()), ("grad", (2,)), ("norm", ()), ("n", (2,)), ("K", ()), ("Fs", (2,)), ("eta", (9,)), ("kappa", (9,)),
              ("rparams", ()), ("omega1", (9,)), ("omega2", (9,)), ("omega3", (9,)))
    _fields_ = [(name, C.POINTER(C.c_double)) for name, _ in FIELDS]


class BcOp(C.Structure):
    _fields_ = [
        ("kind", C.c_int), ("lattice", C.c_int), ("x_begin", C.c_int), ("x_end", C.c_int), ("y_begin", C.c_int),
        ("y_end", C.c_int), ("dst_q", C.c_int), ("src_q", C.c_int), ("src_mode", C.c_int), ("src_a", C.c_int),
        ("src_b", C.c_int), ("coef", C.c_double), ("cst", C.c_double), ("uw", C.c_double * 2), ("rho_bc", C.c_double),
        ("per_row", dp),
    ]


class Params(C.Structure):
    _fields_ = [
        ("flow_nu", C.c_double), ("flow_u", C.c_double), ("flow_l", C.c_double), ("flow_rho_0", C.c_double),
        ("flow_Re", C.c_double),
        ("tau", C.c_double), ("omega", C.c_double), ("Re", C.c_double), ("nu", C.c_double), ("dx", C.c_double),
        ("dt", C.c_double), ("u", C.c_double),
        ("l", C.c_int), ("T", C.c_int), ("X", C.c_int), ("Y", C.c_int),
        ("has_simulation", C.c_int), ("stop_time", C.c_double), ("snapshot_period", C.c_double),
        ("total_steps", C.c_int), ("snapshot_steps", C.c_int), ("total_snapshots", C.c_int),
        ("file_prefix", C.c_char * 256),
    ]


class Colour(C.Structure):
    _fields_ = [
        ("rho_0", C.c_double), ("alpha", C.c_double), ("A", C.c_double), ("nu", C.c_double), ("mu", C.c_double),
        ("beta", C.c_double), ("cs2", C.c_double), ("ics2", C.c_double), ("rlx", C.c_double),
        ("phi", C.c_double * 9), ("eta", C.c_double * 9),
    ]


class TwoPhaseParams(C.Structure):
    _fields_ = [
        ("rows", C.c_int), ("columns", C.c_int), ("time_steps", C.c_int), ("nr_snapshots", C.c_int),
        ("period_snapshots", C.c_int), ("has_general", C.c_int), ("sigma", C.c_double),
        ("gravity_magnitude", C.c_double), ("name", C.c_char * 256),
    ]


EXPORTS = [
    "lbm_last_error", "lbm_version", "lbm_config_default", "lbm_create", "lbm_destroy", "lbm_bc_op_default",
    "lbm_bc_clear", "lbm_bc_add", "lbm_bc_add_solid", "lbm_bc_commit", "lbm_bc_get_mask", "lbm_set_f", "lbm_get_f", "lbm_get_moments",
    "lbm_get_phase", "lbm_set_u", "lbm_init_equilibrium", "lbm_init_two_phase", "lbm_ibm_set_markers",
    "lbm_ibm_get_roi", "lbm_ibm_get_force", "lbm_ibm_force", "lbm_step", "lbm_synchronize", "lbm_last_step_ms",
    "lbm_kernel_launches", "lbm_get_stream", "lbm_use_graph", "lbm_comm_unique_id", "lbm_comm_init",
    "lbm_link_neighbours", "lbm_decompose_rows", "lbm_calc_rho", "lbm_calc_u", "lbm_calc_incomp_u",
    "lbm_equilibrium", "lbm_incomp_equilibrium", "lbm_collision", "lbm_advect", "lbm_differential",
    "lbm_differential3", "lbm_params_from_toml", "lbm_colour_from_toml", "lbm_two_phase_from_toml",
    "lbm_markers_from_toml", "lbm_preset_poiseuille", "lbm_preset_specular_channel", "lbm_preset_free_stream",
    "lbm_preset_sedimentation", "lbm_preset_mrtcg", "lbm_preset_rk", "lbm_preset_periodic",
    "lbm_profile_enable", "lbm_profile_read", "lbm_step_group", "lbm_save_pt", "lbm_snapshot_async", "lbm_snapshot_wait", "lbm_set_moments", "lbm_get_interfacial_tension", "lbm_link_face", "lbm_set_force_region",
    "lbm_rk_diagnostics", "lbm_comm_check", "lbm_comm_share", "lbm_row_split", "lbm_comm_init_blocks", "lbm_link_face_rank", "lbm_comm_faces_commit",
    "lbm_body_force_record", "lbm_body_force_read", "lbm_body_force_stop",
]
PROF_INTERIOR, PROF_BOUNDARY, PROF_FIXUP, PROF_GHOST, PROF_IBM, PROF_MOMENTS, PROF_EARLY = range(7)

_lib = None


def load():
    """Load liblbm_b200.so; raises if it has not been built (python __graft_entry__.py / make)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C lattice-boltzmann-method_b200` "
                "(there is no CPU fallback for the lattice-Boltzmann step)"
            )
        _lib = C.CDLL(LIB_PATH)
        _lib.lbm_last_error.restype = C.c_char_p
        _lib.lbm_version.restype = C.c_char_p
        _lib.lbm_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
        for name in ("lbm_destroy", "lbm_bc_clear", "lbm_bc_commit", "lbm_synchronize"):
            getattr(_lib, name).argtypes = [C.c_void_p]
        _lib.lbm_bc_add.argtypes = [C.c_void_p, C.POINTER(BcOp)]
        _lib.lbm_bc_add_solid.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_ubyte), C.c_int, C.c_int]
        _lib.lbm_bc_get_mask.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int32)]
        _lib.lbm_set_f.argtypes = [C.c_void_p, C.c_int, dp]
        _lib.lbm_get_f.argtypes = [C.c_void_p, C.c_int, dp]
        _lib.lbm_get_moments.argtypes = [C.c_void_p, C.c_int, dp, dp]
        _lib.lbm_get_phase.argtypes = [C.c_void_p, dp, dp, dp]
        _lib.lbm_snapshot_async.argtypes = [C.c_void_p, C.c_int, dp, dp, dp]
        _lib.lbm_snapshot_wait.argtypes = [C.c_void_p]
        _lib.lbm_save_pt.argtypes = [C.c_char_p, dp, C.POINTER(C.c_longlong), C.c_int]
        _lib.lbm_set_u.argtypes = [C.c_void_p, dp]
        _lib.lbm_rk_diagnostics.argtypes = [C.c_void_p, C.c_double, C.POINTER(RkDiag)]
        _lib.lbm_set_moments.argtypes = [C.c_void_p, dp, dp]
        _lib.lbm_get_interfacial_tension.argtypes = [C.c_void_p, dp]
        _lib.lbm_init_equilibrium.argtypes = [C.c_void_p, C.c_int, C.c_int, dp, dp]
        _lib.lbm_init_two_phase.argtypes = [C.c_void_p, dp, dp, dp]
        _lib.lbm_ibm_set_markers.argtypes = [C.c_void_p, dp, dp, C.c_int, C.c_int]
        _lib.lbm_ibm_get_roi.argtypes = [C.c_void_p, C.POINTER(C.c_long)]
        _lib.lbm_ibm_get_force.argtypes = [C.c_void_p, dp]
        _lib.lbm_ibm_force.argtypes = [C.c_void_p, dp, dp, dp]
        _lib.lbm_body_force_record.argtypes = [C.c_void_p, C.POINTER(C.c_ubyte), C.c_int, C.c_int, C.c_int]
        _lib.lbm_body_force_read.argtypes = [C.c_void_p, dp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_longlong)]
        _lib.lbm_body_force_stop.argtypes = [C.c_void_p]
        _lib.lbm_step.argtypes = [C.c_void_p, C.c_int]
        _lib.lbm_last_step_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        _lib.lbm_kernel_launches.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
        _lib.lbm_get_stream.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        _lib.lbm_use_graph.argtypes = [C.c_void_p, C.c_int]
        _lib.lbm_profile_enable.argtypes = [C.c_void_p, C.c_int]
        _lib.lbm_profile_read.argtypes = [C.c_void_p, C.c_int, dp, C.POINTER(C.c_longlong)]
        _lib.lbm_row_split.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        _lib.lbm_comm_unique_id.argtypes = [C.c_char_p]
        _lib.lbm_comm_init.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int]
        _lib.lbm_comm_share.argtypes = [C.c_void_p, C.c_void_p]
        _lib.lbm_comm_init_blocks.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int]
        _lib.lbm_link_face_rank.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        _lib.lbm_comm_faces_commit.argtypes = [C.c_void_p]
        _lib.lbm_link_neighbours.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.lbm_link_face.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
        _lib.lbm_set_force_region.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double]
        _lib.lbm_step_group.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int]
        _lib.lbm_decompose_rows.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        _lib.lbm_calc_rho.argtypes = [dp, C.c_int, C.c_int, dp]
        _lib.lbm_calc_u.argtypes = [dp, dp, C.c_int, C.c_int, dp]
        _lib.lbm_calc_incomp_u.argtypes = [dp, C.c_int, C.c_int, dp]
        _lib.lbm_equilibrium.argtypes = [dp, dp, C.c_int, C.c_int, dp]
        _lib.lbm_incomp_equilibrium.argtypes = [dp, dp, C.c_int, C.c_int, dp]
        _lib.lbm_collision.argtypes = [dp, dp, C.c_double, C.c_int, C.c_int, dp]
        _lib.lbm_advect.argtypes = [dp, C.c_int, C.c_int, dp]
        _lib.lbm_differential.argtypes = [dp, C.c_int, C.c_int, dp, dp]
        _lib.lbm_differential3.argtypes = [dp, C.c_int, C.c_int, dp, dp]
        _lib.lbm_params_from_toml.argtypes = [C.c_char_p, C.c_int, C.POINTER(Params)]
        _lib.lbm_colour_from_toml.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(Colour)]
        _lib.lbm_two_phase_from_toml.argtypes = [C.c_char_p, C.c_int, C.POINTER(TwoPhaseParams)]
        _lib.lbm_markers_from_toml.argtypes = [C.c_char_p, C.c_char_p, dp, dp, C.POINTER(C.c_int)]
        _lib.lbm_preset_poiseuille.argtypes = [C.c_void_p, C.c_double, C.c_double]
        _lib.lbm_preset_specular_channel.argtypes = [C.c_void_p, C.c_double, C.c_double]
        _lib.lbm_preset_free_stream.argtypes = [C.c_void_p, C.c_double, C.c_double]
        _lib.lbm_preset_sedimentation.argtypes = [C.c_void_p, C.c_double, dp, C.c_int, C.c_int, C.c_int]
        for name in ("lbm_preset_mrtcg", "lbm_preset_rk", "lbm_preset_periodic"):
            getattr(_lib, name).argtypes = [C.c_void_p]
    return _lib


def _chk(status):
    if status != OK:
        raise LbmError(status, load().lbm_last_error().decode())


def _in(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(dp)


def _shaped(a, shape, what):
    """contiguous fp64 view of `a` and its pointer; the C ABI takes raw pointers, so a wrong shape (a global array handed
    to a slab, a short vector) would make the library read host memory out of bounds — refuse it here"""
    a, p = _in(a)
    if a.size != int(np.prod(shape)) or (a.ndim == len(shape) and a.shape != tuple(shape)):
        raise ValueError(f"{what}: expected shape {tuple(shape)}, got {a.shape}")
    return a, p


def version():
    return load().lbm_version().decode()


def default_config(**kw):
    cfg = Config()
    load().lbm_config_default(C.byref(cfg))
    for k, v in kw.items():
        if k == "Fg":
            cfg.Fg[0], cfg.Fg[1] = v
        elif k in ("red", "blue"):
            cd = getattr(cfg, k)
            for kk, vv in v.items():
                setattr(cd, kk, vv)
        else:
            setattr(cfg, k, v)
    if cfg.x1 == 0:
        cfg.x1 = cfg.X
    return cfg


def bc_op(_rows=None, **kw):
    op = BcOp()
    load().lbm_bc_op_default(C.byref(op))
    keep = None
    for k, v in kw.items():
        if k == "uw":
            op.uw[0], op.uw[1] = v
        elif k == "per_row":
            keep, ptr = _in(v) if _rows is None else _shaped(v, (_rows,), "bc_add per_row (one value per GLOBAL row)")
            op.per_row = ptr
        else:
            setattr(op, k, v)
    op._keep = keep
    return op


class Domain:
    """One slab on one GPU (the reference's `struct domain`, src/domain.hpp:5-15)."""

    def __init__(self, cfg):
        self.lib = load()
        self.cfg = cfg
        self.h = C.c_void_p()
        _chk(self.lib.lbm_create(C.byref(cfg), C.byref(self.h)))
        self.Xl = cfg.x1 - cfg.x0
        self.Y = cfg.Y

    def close(self):
        if self.h:
            self.lib.lbm_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- boundary rules
    def bc_clear(self):
        _chk(self.lib.lbm_bc_clear(self.h))

    def bc_add(self, **kw):
        op = bc_op(_rows=self.cfg.X, **kw)
        _chk(self.lib.lbm_bc_add(self.h, C.byref(op)))

    def bc_add_solid(self, solid, lattice=0):
        """half-way bounce-back around the non-zero nodes of the GLOBAL {X,Y} mask (staircase body)"""
        m = np.ascontiguousarray(solid, dtype=np.uint8)
        if m.shape != (self.cfg.X, self.cfg.Y):
            raise ValueError("solid mask must have the global shape {X,Y}")
        _chk(self.lib.lbm_bc_add_solid(self.h, lattice, m.ctypes.data_as(C.POINTER(C.c_ubyte)), m.shape[0], m.shape[1]))

    def bc_commit(self):
        _chk(self.lib.lbm_bc_commit(self.h))

    def bc_mask(self, lattice=0):
        m = np.zeros((self.Xl, self.Y, 9), dtype=np.int32)
        _chk(self.lib.lbm_bc_get_mask(self.h, lattice, m.ctypes.data_as(C.POINTER(C.c_int32))))
        return m

    # ---- the reference drivers' rule lists
    def preset_periodic(self):
        _chk(self.lib.lbm_preset_periodic(self.h))

    def preset_poiseuille(self, rho_in, rho_out):
        _chk(self.lib.lbm_preset_poiseuille(self.h, rho_in, rho_out))

    def preset_specular_channel(self, rho_in, rho_out):
        _chk(self.lib.lbm_preset_specular_channel(self.h, rho_in, rho_out))

    def preset_free_stream(self, uwx, uwy=0.0):
        _chk(self.lib.lbm_preset_free_stream(self.h, uwx, uwy))

    def preset_sedimentation(self, u_lb, C_w, R23, C28, C38):
        a, p = _shaped(C_w, (self.cfg.X,), "preset_sedimentation C_w (one value per GLOBAL row)")
        _chk(self.lib.lbm_preset_sedimentation(self.h, u_lb, p, R23, C28, C38))

    def preset_mrtcg(self):
        _chk(self.lib.lbm_preset_mrtcg(self.h))

    def preset_rk(self):
        _chk(self.lib.lbm_preset_rk(self.h))

    # ---- state
    def set_f(self, f, lattice=0):
        a, p = _shaped(f, (self.Xl, self.Y, 9), "set_f")
        _chk(self.lib.lbm_set_f(self.h, lattice, p))

    def get_f(self, lattice=0):
        out = np.empty((self.Xl, self.Y, 9))
        _chk(self.lib.lbm_get_f(self.h, lattice, out.ctypes.data_as(dp)))
        return out

    def get_moments(self, lattice=0):
        rho = np.empty((self.Xl, self.Y, 1)); u = np.empty((self.Xl, self.Y, 2))
        _chk(self.lib.lbm_get_moments(self.h, lattice, rho.ctypes.data_as(dp), u.ctypes.data_as(dp)))
        return rho, u

    def snapshot_async(self, rho=None, u=None, phase=None, lattice=0):
        """rho/u/phase: preallocated (ideally pinned) float64 arrays the copy stream fills; valid after snapshot_wait()"""
        ptr = lambda a: a.ctypes.data_as(dp) if a is not None else None
        for a in (rho, u, phase):
            assert a is None or (a.dtype == np.float64 and a.flags["C_CONTIGUOUS"])
        _chk(self.lib.lbm_snapshot_async(self.h, lattice, ptr(rho), ptr(u), ptr(phase)))

    def snapshot_wait(self):
        _chk(self.lib.lbm_snapshot_wait(self.h))

    def get_phase(self):
        ph = np.empty((self.Xl, self.Y)); rr = np.empty((self.Xl, self.Y)); rb = np.empty((self.Xl, self.Y))
        _chk(self.lib.lbm_get_phase(self.h, ph.ctypes.data_as(dp), rr.ctypes.data_as(dp), rb.ctypes.data_as(dp)))
        return ph, rr, rb

    def rk_diagnostics(self, sigma=5e-3):
        """the fields test/rk_static_droplet_test.cpp snapshots at the top of an iteration, of the current state"""
        out = {name: np.empty((self.Xl, self.Y) + tail) for name, tail in RkDiag.FIELDS}
        arg = RkDiag(**{name: a.ctypes.data_as(dp) for name, a in out.items()})
        _chk(self.lib.lbm_rk_diagnostics(self.h, C.c_double(sigma), C.byref(arg)))
        return out

    def comm_check(self):
        _chk(self.lib.lbm_comm_check(self.h))

    def set_u(self, u):
        a, p = _shaped(u, (self.Xl, self.Y, 2), "set_u")
        _chk(self.lib.lbm_set_u(self.h, p))

    def init_equilibrium(self, rho, u, kind=EQ_INCOMPRESSIBLE, lattice=0):
        r, rp = _shaped(rho, (self.Xl, self.Y, 1), "init_equilibrium rho"); uu, up = _shaped(u, (self.Xl, self.Y, 2), "init_equilibrium u")
        _chk(self.lib.lbm_init_equilibrium(self.h, lattice, kind, rp, up))

    def get_interfacial_tension(self):
        out = np.zeros((self.cfg.x1 - self.cfg.x0, self.cfg.Y, 2))
        _chk(self.lib.lbm_get_interfacial_tension(self.h, out.ctypes.data_as(dp)))
        return out

    def set_moments(self, rho, u):
        """MODEL_KBC: m0 / m1 the first step after an import uses (the ulbm drivers' members)"""
        r, rp = _shaped(rho, (self.Xl, self.Y, 1), "set_moments rho"); uu, up = _shaped(u, (self.Xl, self.Y, 2), "set_moments u")
        _chk(self.lib.lbm_set_moments(self.h, rp, up))

    def init_two_phase(self, rho_r, rho_b, u):
        a, ap = _shaped(rho_r, (self.Xl, self.Y), "init_two_phase rho_r"); b, bp = _shaped(rho_b, (self.Xl, self.Y), "init_two_phase rho_b")
        c, cp = _shaped(u, (self.Xl, self.Y, 2), "init_two_phase u")
        _chk(self.lib.lbm_init_two_phase(self.h, ap, bp, cp))

    # ---- immersed boundary
    def ibm_set_markers(self, xs, ys, m_max=5):
        a, ap = _in(xs); b, bp = _in(ys)
        if a.ndim != 1 or a.shape != b.shape:
            raise ValueError(f"ibm_set_markers: xs and ys must be vectors of one length, got {a.shape} and {b.shape}")
        _chk(self.lib.lbm_ibm_set_markers(self.h, ap, bp, len(a), m_max))

    def ibm_roi(self):
        roi = (C.c_long * 4)()
        _chk(self.lib.lbm_ibm_get_roi(self.h, roi))
        return tuple(int(v) for v in roi)

    def ibm_get_force(self):
        r0, r1, c0, c1 = self.ibm_roi()
        F = np.empty((r1 - r0, c1 - c0, 2))
        _chk(self.lib.lbm_ibm_get_force(self.h, F.ctypes.data_as(dp)))
        return F

    def ibm_force(self, u, rho):
        r0, r1, c0, c1 = self.ibm_roi()
        F = np.empty((r1 - r0, c1 - c0, 2))
        a, ap = _shaped(u, (self.Xl, self.Y, 2), "ibm_force u"); b, bp = _shaped(rho, (self.Xl, self.Y, 1), "ibm_force rho")
        _chk(self.lib.lbm_ibm_force(self.h, ap, bp, F.ctypes.data_as(dp)))
        return F

    # ---- force on a body, recorded on the device every step
    def body_force_record(self, solid=None, capacity=4096):
        """record the force on the bounce-back body of the GLOBAL {X,Y} mask `solid` (as given to bc_add_solid, after
        bc_commit), or with solid=None on the immersed body of ibm_set_markers; the last `capacity` steps are kept"""
        if solid is None:
            _chk(self.lib.lbm_body_force_record(self.h, None, self.cfg.X, self.cfg.Y, int(capacity)))
        else:
            m = np.ascontiguousarray(solid, dtype=np.uint8)
            if m.shape != (self.cfg.X, self.cfg.Y):
                raise ValueError("solid mask must have the global shape {X,Y}")
            _chk(self.lib.lbm_body_force_record(self.h, m.ctypes.data_as(C.POINTER(C.c_ubyte)), m.shape[0], m.shape[1],
                                                int(capacity)))
        self._bf_capacity = int(capacity)

    def body_force(self, max_steps=None):
        """(F, first_step): F {n,2} float64, the force on the body (axis 0, axis 1) of the last n recorded steps in step
        order, first_step the index of F[0] counted from body_force_record.  Synchronises the domain."""
        cap = getattr(self, "_bf_capacity", 0)
        m = cap if max_steps is None else int(max_steps)
        F = np.empty((max(m, 1), 2))
        n = C.c_int(); first = C.c_longlong()
        _chk(self.lib.lbm_body_force_read(self.h, F.ctypes.data_as(dp), m, C.byref(n), C.byref(first)))
        return F[:n.value].copy(), first.value

    def body_force_stop(self):
        _chk(self.lib.lbm_body_force_stop(self.h))
        self._bf_capacity = 0

    # ---- stepping
    def step(self, n=1):
        _chk(self.lib.lbm_step(self.h, int(n)))

    def synchronize(self):
        _chk(self.lib.lbm_synchronize(self.h))

    def last_step_ms(self):
        ms = C.c_float()
        _chk(self.lib.lbm_last_step_ms(self.h, C.byref(ms)))
        return ms.value

    def kernel_launches(self):
        n = C.c_longlong()
        _chk(self.lib.lbm_kernel_launches(self.h, C.byref(n)))
        return n.value

    def stream(self):
        s = C.c_void_p()
        _chk(self.lib.lbm_get_stream(self.h, C.byref(s)))
        return s.value

    def profile_enable(self, enable=True):
        _chk(self.lib.lbm_profile_enable(self.h, 1 if enable else 0))

    def profile_read(self, prof_class):
        ms = C.c_double(); n = C.c_longlong()
        _chk(self.lib.lbm_profile_read(self.h, prof_class, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def row_split(self):
        """(early rows, bulk rows) of the single-phase step's two interior launches"""
        a, b = C.c_int(), C.c_int()
        _chk(self.lib.lbm_row_split(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def use_graph(self, enable=True):
        _chk(self.lib.lbm_use_graph(self.h, 1 if enable else 0))

    # ---- multi-GPU
    def comm_init(self, unique_id, n_ranks, rank):
        _chk(self.lib.lbm_comm_init(self.h, unique_id, n_ranks, rank))

    def comm_init_blocks(self, unique_id, n_ranks, rank):
        """join the communicator of independent blocks bound across column faces (one block per process)"""
        _chk(self.lib.lbm_comm_init_blocks(self.h, unique_id, n_ranks, rank))

    def link_face_rank(self, side, row_begin, n_rows, peer_rank, peer_row_begin):
        """link_face with the facing block on another rank (call on the reading rank)"""
        _chk(self.lib.lbm_link_face_rank(self.h, side, row_begin, n_rows, peer_rank, peer_row_begin))

    def comm_faces_commit(self):
        _chk(self.lib.lbm_comm_faces_commit(self.h))

    def comm_share(self, member):
        """join the ring `member` belongs to, on its communicator"""
        _chk(self.lib.lbm_comm_share(self.h, member.h))

    def link_face(self, side, row_begin, n_rows, other, other_row_begin):
        """bind rows [row_begin, row_begin + n_rows) of the first (side 0) / last (side 1) column to the facing column of `other`"""
        _chk(self.lib.lbm_link_face(self.h, side, row_begin, n_rows, other.h, other_row_begin))

    def set_force_region(self, x_begin, x_end, y_begin, y_end, Fx, Fy, ics2=3.0, ics4=9.0):
        _chk(self.lib.lbm_set_force_region(self.h, x_begin, x_end, y_begin, y_end, Fx, Fy, ics2, ics4))

    def link(self, lower, upper):
        _chk(self.lib.lbm_link_neighbours(self.h, lower.h if lower else None, upper.h if upper else None))


def step_group(domains, n_steps=1):
    """advance linked slabs in lock step"""
    arr = (C.c_void_p * len(domains))(*[d.h for d in domains])
    _chk(load().lbm_step_group(arr, len(domains), int(n_steps)))


def body_force_group(domains, max_steps=None):
    """(F, first_step) of one body over linked slabs: the sum of every slab's part (each records the fluid on its rows)"""
    parts = [d.body_force(max_steps) for d in domains]
    if any(p[1] != parts[0][1] or len(p[0]) != len(parts[0][0]) for p in parts):
        raise ValueError("body_force_group: the slabs' records cover different steps (record on every slab, then step them together)")
    F = parts[0][0].copy()
    for p in parts[1:]:
        F += p[0]
    return F, parts[0][1]


def comm_unique_id():
    buf = C.create_string_buffer(UNIQUE_ID_BYTES)
    _chk(load().lbm_comm_unique_id(buf))
    return buf.raw


def decompose_rows(X, n_ranks, rank):
    a, b = C.c_int(), C.c_int()
    _chk(load().lbm_decompose_rows(X, n_ranks, rank, C.byref(a), C.byref(b)))
    return a.value, b.value


# ---- granular operators (namespace solver, class differential)
def _op_out(shape):
    o = np.empty(shape)
    return o, o.ctypes.data_as(dp)


def calc_rho(f):
    a, p = _in(f); X, Y, _ = a.shape
    o, op = _op_out((X, Y, 1)); _chk(load().lbm_calc_rho(p, X, Y, op)); return o


def calc_u(f, rho):
    a, p = _in(f); r, rp = _in(rho); X, Y, _ = a.shape
    o, op = _op_out((X, Y, 2)); _chk(load().lbm_calc_u(p, rp, X, Y, op)); return o


def calc_incomp_u(f):
    a, p = _in(f); X, Y, _ = a.shape
    o, op = _op_out((X, Y, 2)); _chk(load().lbm_calc_incomp_u(p, X, Y, op)); return o


def equilibrium(u, rho):
    a, p = _in(u); r, rp = _in(rho); X, Y, _ = a.shape
    o, op = _op_out((X, Y, 9)); _chk(load().lbm_equilibrium(p, rp, X, Y, op)); return o


def incomp_equilibrium(u, rho):
    a, p = _in(u); r, rp = _in(rho); X, Y, _ = a.shape
    o, op = _op_out((X, Y, 9)); _chk(load().lbm_incomp_equilibrium(p, rp, X, Y, op)); return o


def collision(f, feq, omega):
    a, p = _in(f); b, bp = _in(feq); X, Y, _ = a.shape
    o, op = _op_out((X, Y, 9)); _chk(load().lbm_collision(p, bp, C.c_double(omega), X, Y, op)); return o


def advect(f):
    a, p = _in(f); X, Y, _ = a.shape
    o, op = _op_out((X, Y, 9)); _chk(load().lbm_advect(p, X, Y, op)); return o


def differential(psi):
    a, p = _in(psi); R, Cc = a.shape
    dx, dxp = _op_out((R, Cc)); dy, dyp = _op_out((R, Cc))
    _chk(load().lbm_differential(p, R, Cc, dxp, dyp)); return dx, dy


def differential3(psi):
    a, p = _in(psi); R, Cc = a.shape
    dx, dxp = _op_out((R, Cc)); dy, dyp = _op_out((R, Cc))
    _chk(load().lbm_differential3(p, R, Cc, dxp, dyp)); return dx, dy


# ---- parameters.toml surface
def save_pt(path, array):
    """torch::save(tensor, path) of the reference drivers: a TorchScript archive holding one fp64 tensor"""
    a = np.ascontiguousarray(array, dtype=np.float64)
    shape = (C.c_longlong * max(a.ndim, 1))(*a.shape)
    _chk(load().lbm_save_pt(os.fsencode(path), a.ctypes.data_as(dp), shape, a.ndim))


def params_from_toml(path, require_simulation=True):
    p = Params()
    _chk(load().lbm_params_from_toml(path.encode(), 1 if require_simulation else 0, C.byref(p)))
    return p


def colour_from_toml(path, table):
    c = Colour()
    _chk(load().lbm_colour_from_toml(path.encode(), table.encode(), C.byref(c)))
    return c


def two_phase_from_toml(path, require_general=False):
    p = TwoPhaseParams()
    _chk(load().lbm_two_phase_from_toml(path.encode(), 1 if require_general else 0, C.byref(p)))
    return p


def markers_from_toml(path, name):
    n = C.c_int(0)
    _chk(load().lbm_markers_from_toml(path.encode(), name.encode(), None, None, C.byref(n)))
    xs = np.empty(n.value); ys = np.empty(n.value)
    _chk(load().lbm_markers_from_toml(path.encode(), name.encode(), xs.ctypes.data_as(dp), ys.ctypes.data_as(dp), C.byref(n)))
    return xs, ys
