"""TEST INFRASTRUCTURE ONLY -- ctypes binding to the parity oracles.

  RefOracle("o2" | "intended")  -> oracle/_ref/libref_*.so : the reference's own sources compiled unmodified
                                   (see oracle/Makefile, oracle/ref_harness.cpp)
  PortOracle()                  -> oracle/liboracle_port.so : the plain-C++ restatement (oracle/port/)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
The product library (liblmot.so) never does.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TRACK_DUMP_DOUBLES = 236

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")


def ref_lib_path(mode: str) -> str:
    return os.path.join(HERE, "_ref", f"libref_{mode}.so")


def have_ref(mode: str = "intended") -> bool:
    return os.path.exists(ref_lib_path(mode))


def _as_pts(points: np.ndarray):
    p = np.ascontiguousarray(points, dtype=np.float32)
    assert p.ndim == 2 and p.shape[1] in (3, 4)
    return p, p.shape[0], p.shape[1]


class _OracleBase:
    """Shared marshalling; `prefix` selects ref_* (reference sources) or port_* (restatement) symbols."""

    def __init__(self, path: str, prefix: str):
        self.lib = C.CDLL(path)
        self.prefix = prefix
        L, p = self.lib, prefix
        self._cell = getattr(L, p + "cell_index"); self._cell.argtypes = [_f32p, C.c_int, C.c_int, _i32p, _i32p]
        self._gr = getattr(L, p + "ground_remove"); self._gr.argtypes = [_f32p, C.c_int, C.c_int, _f32p, C.POINTER(C.c_int), _f32p, C.POINTER(C.c_int)]
        self._pg = getattr(L, p + "polar_grid"); self._pg.argtypes = [_f32p, C.c_int, C.c_int] + [_f32p] * 5 + [_u8p]
        self._cc = getattr(L, p + "component_clustering"); self._cc.argtypes = [_f32p, C.c_int, C.c_int, _i32p, C.POINTER(C.c_int)]
        self._bf = getattr(L, p + "box_fitting"); self._bf.argtypes = [_f32p, C.c_int, C.c_int, _i32p, C.c_int, C.c_int, _f32p, C.POINTER(C.c_int), _f32p]
        self._co = getattr(L, p + "cluster_outputs", None)      # the cluster node's side outputs (reference build only)
        if self._co is not None:
            self._co.argtypes = [_f32p, C.c_int, C.c_int, _i32p, C.c_int, _f32p, C.POINTER(C.c_int), _f64p, C.POINTER(C.c_int), _i32p]
        self._tr = getattr(L, p + "tracker_reset"); self._tr.argtypes = []
        self._tn = getattr(L, p + "tracker_num_tracks"); self._tn.restype = C.c_int
        self._ts = getattr(L, p + "tracker_step")
        self._ts.argtypes = [_f32p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, _f32p, _f64p, _i32p, _u8p, _u8p, _f32p,
                             C.POINTER(C.c_int), C.POINTER(C.c_int)]
        self._td = getattr(L, p + "tracker_dump"); self._td.argtypes = [C.c_int, _f64p]
        self._tl = getattr(L, p + "tracker_load")
        self._tl.argtypes = [C.c_int, _f64p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double]

    # -- ground removal -------------------------------------------------------------------------
    def cell_index(self, points):
        p, n, s = _as_pts(points)
        ch = np.empty(n, np.int32); b = np.empty(n, np.int32)
        self._cell(p, n, s, ch, b)
        return ch, b

    def ground_remove(self, points):
        """-> (elevated (Ne,3), ground (Ng,3)) in input order."""
        p, n, s = _as_pts(points)
        e = np.empty((max(n, 1), 3), np.float32); g = np.empty((max(n, 1), 3), np.float32)
        ne = C.c_int(0); ng = C.c_int(0)
        self._gr(p, n, s, e, C.byref(ne), g, C.byref(ng))
        return e[: ne.value].copy(), g[: ng.value].copy()

    def polar_grid(self, points):
        p, n, s = _as_pts(points)
        out = [np.empty(80 * 120, np.float32) for _ in range(5)]
        isg = np.empty(80 * 120, np.uint8)
        self._pg(p, n, s, *out, isg)
        names = ["minz", "height", "smoothed", "hdiff", "hground"]
        d = {k: v.reshape(80, 120) for k, v in zip(names, out)}
        d["isground"] = isg.reshape(80, 120)
        return d

    # -- clustering / boxes ---------------------------------------------------------------------
    def component_clustering(self, elevated):
        p, n, s = _as_pts(elevated) if len(elevated) else (np.zeros((1, 3), np.float32), 0, 3)
        grid = np.zeros(250 * 250, np.int32); nc = C.c_int(0)
        self._cc(p, n, s, grid, C.byref(nc))
        return grid.reshape(250, 250), nc.value

    def box_fitting(self, elevated, grid, num_cluster, max_boxes: int = 4096):
        p, n, s = _as_pts(elevated) if len(elevated) else (np.zeros((1, 3), np.float32), 0, 3)
        boxes = np.zeros((max_boxes, 8, 3), np.float32); markers = np.zeros((max_boxes, 6), np.float32); nb = C.c_int(0)
        self._bf(p, n, s, np.ascontiguousarray(grid, np.int32).reshape(-1), int(num_cluster), max_boxes, boxes, C.byref(nb), markers)
        return boxes[: nb.value].copy(), markers[: nb.value].copy()

    def cluster_outputs(self, elevated, grid):
        """makeClusteredCloud, setObsMsg, createCostMap -> (clustered (n,3) f32, obstacles (m,4) f64 [x,y,z,cluster], cost_map (50,50) i32)"""
        if self._co is None:
            raise RuntimeError("cluster_outputs is only available from the compiled reference (oracle/_ref)")
        p, n, s = _as_pts(elevated) if len(elevated) else (np.zeros((1, 3), np.float32), 0, 3)
        cap = max(n, 1)
        cl = np.zeros((cap, 3), np.float32); ob = np.zeros((cap, 4), np.float64); cm = np.zeros(2500, np.int32)
        ncl = C.c_int(0); nob = C.c_int(0)
        self._co(p, n, s, np.ascontiguousarray(grid, np.int32).reshape(-1), cap, cl, C.byref(ncl), ob, C.byref(nob), cm)
        return cl[: ncl.value].copy(), ob[: nob.value].copy(), cm.reshape(50, 50)

    # -- tracker --------------------------------------------------------------------------------
    def tracker_reset(self):
        self._tr()

    def tracker_num_tracks(self) -> int:
        return self._tn()

    def tracker_step(self, boxes, timestamp_us, v_gps=0.0, yaw_gps=0.0, cap: int = 16384):
        b = np.ascontiguousarray(boxes, np.float32).reshape(-1, 8, 3)
        m = b.shape[0]
        if m == 0:
            b = np.zeros((1, 8, 3), np.float32)
        tg = np.zeros((cap, 3), np.float32); vy = np.zeros((cap, 2), np.float64); tm = np.zeros(cap, np.int32)
        st = np.zeros(cap, np.uint8); vis = np.zeros(cap, np.uint8); vbb = np.zeros((cap, 8, 3), np.float32)
        nv = C.c_int(0); nt = C.c_int(0)
        self._ts(b, m, float(timestamp_us), float(v_gps), float(yaw_gps), cap, tg, vy, tm, st, vis, vbb, C.byref(nv), C.byref(nt))
        t = nt.value
        return dict(targets=tg[:t].copy(), vandyaw=vy[:t].copy(), track_manage=tm[:t].copy(), is_static=st[:t].copy(),
                    is_vis=vis[:t].copy(), vis_bb=vbb[: nv.value].copy())

    def tracker_dump(self) -> np.ndarray:
        t = self.tracker_num_tracks()
        out = np.zeros((t, TRACK_DUMP_DOUBLES), np.float64)
        row = np.zeros(TRACK_DUMP_DOUBLES, np.float64)
        for i in range(t):
            self._td(i, row)
            out[i] = row
        return out

    def tracker_load(self, dumps, init, timestamp, ego_velo=0.0, ego_yaw=0.0, ego_pre_yaw=0.0, ego_point_yaw=-np.pi / 2):
        d = np.ascontiguousarray(dumps, np.float64).reshape(-1, TRACK_DUMP_DOUBLES)
        if d.shape[0] == 0:
            d2 = np.zeros((1, TRACK_DUMP_DOUBLES), np.float64)
            self._tl(0, d2, int(init), timestamp, ego_velo, ego_yaw, ego_pre_yaw, ego_point_yaw)
        else:
            self._tl(d.shape[0], d, int(init), timestamp, ego_velo, ego_yaw, ego_pre_yaw, ego_point_yaw)


class RefOracle(_OracleBase):
    def __init__(self, mode: str = "intended"):
        assert mode in ("o2", "intended")
        super().__init__(ref_lib_path(mode), "ref_")
        self.mode = mode
        self.lib.ref_build_info.restype = C.c_char_p
        self._time = self.lib.ref_time_detect
        self._time.argtypes = [_f32p, C.c_int, C.c_int, _f64p, C.c_int, _f32p, C.POINTER(C.c_int)]

    def build_info(self) -> str:
        return self.lib.ref_build_info().decode()

    def time_detect(self, points, max_boxes: int = 4096):
        """Run ground->cluster->box once; -> (seconds[3], boxes)."""
        p, n, s = _as_pts(points)
        sec = np.zeros(3, np.float64); boxes = np.zeros((max_boxes, 8, 3), np.float32); nb = C.c_int(0)
        self._time(p, n, s, sec, max_boxes, boxes, C.byref(nb))
        return sec, boxes[: nb.value].copy()


class PortOracle(_OracleBase):
    def __init__(self, mode: str = "intended", path: str | None = None):
        super().__init__(path or os.path.join(HERE, "liboracle_port.so"), "port_")
        self.mode = mode
        self.lib.port_set_rule_mode(0 if mode == "intended" else 1)

    def box_fitting(self, elevated, grid, num_cluster, max_boxes: int = 4096):
        self.lib.port_set_rule_mode(0 if self.mode == "intended" else 1)   # the mode is process-global in the port
        return super().box_fitting(elevated, grid, num_cluster, max_boxes)


def have_port() -> bool:
    return os.path.exists(os.path.join(HERE, "liboracle_port.so"))


def labels_from_clouds(points, elevated, ground) -> np.ndarray:
    """Recover per-point labels (0 dropped, 1 ground, 2 elevated) from the two order-preserving output clouds."""
    p = np.ascontiguousarray(points, np.float32)[:, :3]
    n = len(p)
    lab = np.zeros(n, np.uint8)
    ie = ig = 0
    for i in range(n):
        if ie < len(elevated) and p[i, 0] == elevated[ie, 0] and p[i, 1] == elevated[ie, 1] and p[i, 2] == elevated[ie, 2]:
            lab[i] = 2; ie += 1
        elif ig < len(ground) and p[i, 0] == ground[ig, 0] and p[i, 1] == ground[ig, 1] and p[i, 2] == ground[ig, 2]:
            lab[i] = 1; ig += 1
    assert ie == len(elevated) and ig == len(ground), "clouds are not order-preserving subsequences"
    return lab
