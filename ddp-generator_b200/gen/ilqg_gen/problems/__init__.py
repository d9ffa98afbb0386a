from . import brachi, brachi_hli, car, carhx, cartrack, pend, quad  # noqa: F401

REGISTRY = {"car": car.define, "brachi": brachi.define, "quad": quad.define, "carhx": carhx.define,
            "brachi_hli": brachi_hli.define, "pend": pend.define,
            "cartrack": cartrack.define}
