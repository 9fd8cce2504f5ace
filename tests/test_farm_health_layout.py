"""The farm copy's argument structs and the health constants of include/go1mpc.h match the ctypes binding: a C program compiled
against the header prints sizeof, offsetof / sizeof of every field of Go1FarmColumns and Go1FarmCopy, and every GO1MPC_HEALTH_*
value; health_d is Go1FarmColumns' last field, so existing initialisers stay valid."""
import ctypes
import json
import os
import subprocess

import quadrupedal_loco_b200 as q

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STRUCTS = {"Go1FarmColumns": q.FarmColumns, "Go1FarmCopy": q.FarmCopy}
HEALTH = ["PLAN_OK", "PLAN_INFEASIBLE", "PLAN_FAILED", "BODY_OK", "BODY_INFEASIBLE", "BODY_FAILED", "GRF_OK", "GRF_FAILED",
          "GRF_FALLBACK", "IK_CAP", "NONFINITE", "EVENTS", "ROWS"]


def c_layouts(tmp_path):
    lines = ["#include <stddef.h>", "#include <stdio.h>", '#include "go1mpc.h"', "int main(void) {", '  printf("{");']
    for cname, py in STRUCTS.items():
        lines.append(f'  printf("\\"{cname}\\": {{\\"size\\": %zu, \\"fields\\": {{", sizeof({cname}));')
        for j, (f, _) in enumerate(py._fields_):
            fs = "," if j else ""
            lines.append(f'  printf("{fs}\\"{f}\\": [%zu, %zu]", offsetof({cname}, {f}), sizeof((({cname} *)0)->{f}));')
        lines.append('  printf("}},");')
    lines.append('  printf("\\"health\\": {");')
    for j, n in enumerate(HEALTH):
        fs = "," if j else ""
        lines.append(f'  printf("{fs}\\"{n}\\": %d", (int)GO1MPC_HEALTH_{n});')
    lines += ['  printf("}}\\n");', "  return 0;", "}"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines) + "\n")
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    return json.loads(out)


def test_farm_copy_structs_and_health_rows_match_header(tmp_path):
    got = c_layouts(tmp_path)
    for cname, py in STRUCTS.items():
        c = got[cname]
        assert c["size"] == ctypes.sizeof(py), cname
        for f, _ in py._fields_:
            d = getattr(py, f)
            assert c["fields"][f] == [d.offset, d.size], f"{cname}.{f}: header {c['fields'][f]}, ctypes {[d.offset, d.size]}"
    for n in HEALTH:
        assert got["health"][n] == getattr(q, "HEALTH_" + n), n
    assert got["health"]["ROWS"] == 12 and [got["health"][n] for n in HEALTH[:-1]] == list(range(12))


def test_health_field_is_appended():
    assert [f for f, _ in q.FarmColumns._fields_][-1] == "health_d"
    assert "go1mpc_gait_stack_tick_clocked_health_async" in q.EXPORTED_SYMBOLS
    assert "go1mpc_servo_torque_tick_health_async" in q.EXPORTED_SYMBOLS
