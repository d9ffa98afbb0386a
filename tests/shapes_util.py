"""The test-only problems tests/data/shape_<nx>x<nu>.mac: shapes (nx, nu) no shipped problem has, their library names and a
parameter set under which every input's box binds (tests/test_gpu_shapes.py, tests/test_mmex_gateway.py; built by
__graft_entry__.build_shape_problems into ddp-generator_b200/build_shapes/)."""
import numpy as np

LANE = ((4, 1), (3, 4), (6, 3))          # one lane per problem: k_backpass_split and k_backpass
COOP = ((7, 5), (10, 9), (16, 9))        # the warp-cooperative k_backpass_warp (nx > 6)
SHAPES = LANE + COOP


def name_of(shape):
    return f"shape_{shape[0]}x{shape[1]}"


def params_of(shape, dt=0.25):
    """The odd inputs get the tighter box: with three or more inputs, a clamped input sits between two free ones."""
    nx, nu = shape
    lim = [0.25 if j % 2 else 0.6 for j in range(nu)]
    return {"dt": [dt], "a": list(0.4 + 0.6 * np.arange(nx) / nx), "b": [1.0] * nu, "kxu": [0.5], "kuu": [0.3], "cx": [0.2] * nx,
            "cu": [0.05] * nu, "cf": [5.0] * nx, "ulo": [-v for v in lim], "uhi": lim}
