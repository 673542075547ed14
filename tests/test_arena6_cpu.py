"""CPU suite: the six-player arena's result struct (az_arena6_results) as the Python binding declares it agrees with the C header,
field by field in order, and in size."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_fields():
    text = open(os.path.join(ROOT, "include", "az_b200.h")).read()
    body = re.search(r"typedef struct az_arena6_results \{(.*?)\} az_arena6_results;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        assert decl.startswith("uint64_t "), decl
        for name in decl[len("uint64_t "):].split(","):
            m = re.fullmatch(r"\s*([a-z_]+)\s*(?:\[(\d+)\])?\s*", name)
            fields.append((m.group(1), int(m.group(2)) if m.group(2) else 1))
    return fields


def test_results_layout_agrees_with_header():
    from alphazero_risk_b200 import api
    fields = header_fields()
    assert [f for f, _ in fields] == ["count", "draw", "win", "win_seat", "moves", "sims", "evals", "ticks", "errors"]
    py = [(name, C.sizeof(t) // 8) for name, t in api.AzArena6Results._fields_]
    assert py == fields
    for name, t in api.AzArena6Results._fields_:
        assert getattr(api.AzArena6Results, name).offset % 8 == 0
        assert C.sizeof(t) % C.sizeof(C.c_uint64) == 0
    assert C.sizeof(api.AzArena6Results) == 8 * sum(k for _, k in fields) == 192

