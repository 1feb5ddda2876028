"""Loader for the lane-1 host build with the multi-scene clutter entry point (TEST HARNESS ONLY, see lane1_scenes.cpp)."""
import ctypes as C
import os
import subprocess
import tempfile

from mj_grasp_sim_b200 import lib as mlib

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {}


def build(f64=False):
    so = os.path.join(_HERE, "liblane1_scenes_f64.so" if f64 else "liblane1_scenes_f32.so")
    srcs = [os.path.join(_HERE, "lane1_scenes.cpp"), os.path.join(_HERE, "lane1.cpp")] + mlib._sources()
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(s) for s in srcs):
        # compile to a private file and rename it into place: parallel test workers never load a half-written library
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=_HERE)
        os.close(fd)
        try:
            cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared"] + (["-DMGS_REAL_DOUBLE"] if f64 else []) + [
                "-x", "c++", "-o", tmp, os.path.join(_HERE, "lane1_scenes.cpp")]
            subprocess.check_call(cmd)
            os.replace(tmp, so)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    return so


def sim(model, f64=False):
    so = build(f64)
    if so not in _LIBS:
        L = mlib.bind(C.CDLL(so), prefix="l1_")
        vp, ip, fp, dp, u8p = C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_ubyte)
        L.l1_clutter_scenes_host.argtypes = [vp, C.c_int, C.c_int, C.c_int, dp, ip, C.c_int, fp, fp, C.c_int, ip, C.c_int, dp,
                                             C.POINTER(mlib.MgsRolloutCfg), u8p, ip]
        _LIBS[so] = L
    return mlib.BatchSim(model, lib=_LIBS[so], prefix="l1_")
