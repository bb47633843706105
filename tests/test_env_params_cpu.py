"""Per-env physical parameters: the header's buffer ids and entry point agree with the Python binding (no GPU needed)."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_env_param_buffers_match_the_header():
    from b2sim import _lib
    with open(os.path.join(ROOT, "include", "b2sim.h")) as f:
        header = f.read()
    ids = {name: int(v) for name, v in re.findall(r"\bB2_BUF_([A-Z_]+)\s*=\s*(\d+)", header)}
    assert (ids["BODY_INERTIA"], ids["JOINT_DYNAMICS"], ids["GRAVITY"], ids["COUNT"]) == (20, 21, 22, 23)
    for name in ("BODY_INERTIA", "JOINT_DYNAMICS", "GRAVITY"):
        assert getattr(_lib, "BUF_" + name) == ids[name]
    assert "int b2sim_enable_env_params(b2sim* s, int model, int enable);" in header
    assert _lib.SYMBOLS["b2sim_enable_env_params"][1] == [_lib._vp, _lib._i, _lib._i]
