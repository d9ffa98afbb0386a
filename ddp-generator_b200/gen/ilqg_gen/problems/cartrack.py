"""Car tracking a reference path (authored here): the dynamics and input limits of the car-parking problem (car.py), with
the parking cost replaced by a cost on the distance to a time-indexed reference point xr[k], yr[k].  In a receding-horizon
loop the reference moves with the plan, so every problem of a batch can follow its own path (per-problem tracks)."""
import sympy as sp

from ..problem import Problem
from .car import sqrt_abs


def define():
    P = Problem("CarTrack")
    x_, y_, t, v = P.states("x_ y_ t v")
    w, a = P.inputs("w a")
    d = P.param("d")
    h = P.param("h")
    cu = P.param_array("cu", 2)
    cx = P.param_array("cx", 2)
    px = P.param_array("px", 2)
    cf = P.param_array("cf", 2)
    limW = P.param_array("limW", 2)
    limA = P.param_array("limA", 2)
    xr = P.param_k("xr")
    yr = P.param_k("yr")

    s = P.def_aux("s", d + h * v * sp.cos(w) - sp.sqrt(d**2 - (h * v * sp.sin(w)) ** 2))
    P.f[x_] = x_ + s * sp.cos(t)
    P.f[y_] = y_ + s * sp.sin(t)
    P.f[t] = t + sp.asin(sp.sin(w) * h * v / d)
    P.f[v] = v + h * a

    # the final cost reads xr, yr at k = N, like brachi_hli's hfe reads ymin[N]
    P.F = cf[0] * sqrt_abs(x_ - xr, px[0]) + cf[1] * sqrt_abs(y_ - yr, px[1])
    P.L = cu[0] * w**2 + cu[1] * a**2 + cx[0] * sqrt_abs(x_ - xr, px[0]) + cx[1] * sqrt_abs(y_ - yr, px[1])

    P.h = [-w + limW[0], w - limW[1], -a + limA[0], a - limA[1]]
    return P
