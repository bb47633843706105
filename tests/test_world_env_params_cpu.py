"""Per-env free-body and friction rows: the header's entry points agree with the Python binding, and the new rows come as
views of their own, not as new buffer ids (no GPU needed)."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header():
    with open(os.path.join(ROOT, "include", "b2sim.h")) as f:
        return f.read()


def test_world_row_entry_points_match_the_binding():
    from b2sim import _lib
    text = header()
    for name in ("b2sim_enable_free_body_params", "b2sim_enable_shape_friction"):
        assert f"int {name}(b2sim* s, int model, int enable, b2_buffer* out);" in text
        res, args = _lib.SYMBOLS[name]
        assert res is _lib._i
        assert args[:3] == [_lib._vp, _lib._i, _lib._i]
        assert args[3]._type_ is _lib.Buffer


def test_buffer_ids_are_unchanged():
    from b2sim import _lib
    ids = {name: int(v) for name, v in re.findall(r"\bB2_BUF_([A-Z_]+)\s*=\s*(\d+)", header())}
    assert ids["COUNT"] == 23 and len(ids) == 24
    assert sorted(v for k, v in ids.items() if k != "COUNT") == list(range(23))
    for name, v in ids.items():
        if name != "COUNT":
            assert getattr(_lib, "BUF_" + name) == v
