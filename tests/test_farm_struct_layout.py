"""The ctypes mirrors of the farm's argument structs match include/go1mpc.h: a C program compiled against the header with the
host compiler prints sizeof, and offsetof / sizeof of every field, of Go1GaitStackTick, Go1GaitStackClockedTick,
Go1GaitStackReset and Go1ServoTorqueTick; each must equal the ctypes structure's.  Guards the fields appended for device
inputs, and every older field, against ABI drift (a field missing from the header fails the compile)."""
import ctypes
import json
import os
import subprocess

import quadrupedal_loco_b200 as q

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STRUCTS = {"Go1GaitStackTick": q.GaitStackTick, "Go1GaitStackClockedTick": q.GaitStackClockedTick,
           "Go1GaitStackReset": q.GaitStackReset, "Go1ServoTorqueTick": q.ServoTorqueTick}


def c_layouts(tmp_path):
    lines = ["#include <stddef.h>", "#include <stdio.h>", '#include "go1mpc.h"', "int main(void) {", '  printf("{");']
    for i, (cname, py) in enumerate(STRUCTS.items()):
        sep = "," if i else ""
        lines.append(f'  printf("{sep}\\"{cname}\\": {{\\"size\\": %zu, \\"fields\\": {{", sizeof({cname}));')
        for j, (f, _) in enumerate(py._fields_):
            fs = "," if j else ""
            lines.append(f'  printf("{fs}\\"{f}\\": [%zu, %zu]", offsetof({cname}, {f}), sizeof((({cname} *)0)->{f}));')
        lines.append('  printf("}}");')
    lines += ['  printf("}\\n");', "  return 0;", "}"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines) + "\n")
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    return json.loads(out)


def test_farm_structs_match_header(tmp_path):
    got = c_layouts(tmp_path)
    for cname, py in STRUCTS.items():
        c = got[cname]
        assert c["size"] == ctypes.sizeof(py), cname
        for f, _ in py._fields_:
            d = getattr(py, f)
            assert c["fields"][f] == [d.offset, d.size], f"{cname}.{f}: header {c['fields'][f]}, ctypes {[d.offset, d.size]}"


def test_device_input_fields_are_appended():
    """The device inputs come after every field the structs had before, so existing initialisers and field orders stay valid."""
    tail = {"Go1GaitStackTick": ["sensor_d", "cmd_d", "start_d"], "Go1GaitStackClockedTick": ["sensor_d", "cmd_d", "start_d"],
            "Go1GaitStackReset": ["reset_d"], "Go1ServoTorqueTick": ["reset_d"]}
    for cname, py in STRUCTS.items():
        names = [f for f, _ in py._fields_]
        assert names[-len(tail[cname]):] == tail[cname], cname
