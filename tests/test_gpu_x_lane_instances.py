"""Every compiled instance of the lane kernel against the oracle on one GPU.

launch_pass runs each lane pass on one of the compiled lane_kernel<E, LN, TPL> instances: the compile-time-geometry ("fast")
instances of its B2_INST list and the generic instances {16, 8, 4} x {4, 2}.  Each family runs different operator code (the
*_fast operators and OP_BANDC / OP_PREBAND on fast instances, LD_STENCIL loads on generic ones) with its own scan-layout
coefficient vectors.  With default settings one GPU reaches only some of them (DEFAULT_LAYOUTS); the rest are reached through
the geometry knobs B2_E, B2_LN and B2_NOFAST, which make_cfg reads when a space is created.  CASES reaches each of those
instances, checks that the knobs really chose it (Space2.lane_layout) and bounds every operator and a 2-step Navier2D run at
1e-12 relative -- far tighter than the 1e-10 of the other suites, which a 1000x loss of accuracy would still pass.

B2_CHW (sub-chunk width, read by make_cfg) gets the same treatment.  B2_NOTMA and B2_LDTHREADS are read once when the library
loads, so FRESH_CASES run in a child process.

The CPU tests of this file check that CASES plus DEFAULT_LAYOUTS add up to exactly the compiled instance set, and run the
same checks in the SIMT emulator of tests/emu for the cases whose lanes are at most 1025 points."""
import json
import os
import re
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-12
KNOBS = ("B2_E", "B2_LN", "B2_NOFAST", "B2_CHW", "B2_SMEMCAP", "B2_NOTMA", "B2_LDTHREADS")
CH, CD, CN, CDN, R2C = 0, 1, 2, 3, 4


def lay(e, ln, tpl, fast):
    return (e, ln, tpl, fast)


# case: knobs; spaces as ((kind0, n0, kind1, n1), (layout of orient 0 = lanes along axis 1, layout of orient 1 = lanes along
# axis 0)) with layout = (E, LN, TPL, fast); Navier2D runs as (nx, ny, periodic, bc); chw: the sub-chunk width the knob forces
CASES = {
    "E16-T8": dict(env={"B2_E": "16"},
                   spaces=[((CD, 257, CN, 257), (lay(16, 4, 8, 1), lay(16, 4, 8, 1))),
                           ((R2C, 256, CD, 257), (lay(16, 4, 8, 1), lay(16, 4, 8, 1)))],
                   navier=[(257, 257, False, "rbc"), (256, 257, True, "rbc")]),
    "E16-T16": dict(env={"B2_E": "16"},
                    spaces=[((CD, 513, CN, 65), (lay(4, 4, 8, 1), lay(16, 4, 16, 1))),
                            ((CN, 65, CD, 513), (lay(16, 4, 16, 1), lay(4, 4, 8, 1)))],
                    navier=[(513, 129, False, "rbc")]),
    "E16-T32": dict(env={"B2_E": "16"},
                    spaces=[((CD, 1025, CN, 129), (lay(8, 4, 8, 1), lay(16, 4, 32, 1))),
                            ((R2C, 1024, CD, 65), (lay(4, 4, 8, 1), lay(16, 4, 32, 1)))],
                    navier=[]),
    "E4-T16": dict(env={"B2_E": "4"},
                   spaces=[((CD, 129, CN, 129), (lay(4, 4, 16, 1), lay(4, 4, 16, 1))),
                           ((R2C, 128, CD, 129), (lay(4, 4, 16, 1), lay(4, 4, 16, 1))),
                           ((CN, 129, CDN, 129), (lay(4, 4, 16, 1), lay(4, 4, 16, 1)))],
                   navier=[(129, 129, False, "rbc"), (128, 129, True, "rbc"), (129, 129, False, "hc")]),
    "E4-T32": dict(env={"B2_E": "4"},
                   spaces=[((CN, 257, CD, 257), (lay(4, 4, 32, 1), lay(4, 4, 32, 1)))],
                   navier=[(257, 257, False, "rbc")]),
    "LN2-T128": dict(env={"B2_LN": "2"},
                     spaces=[((CD, 4097, CN, 65), (lay(4, 4, 8, 1), lay(16, 2, 128, 1))),
                             ((R2C, 4096, CD, 65), (lay(4, 4, 8, 1), lay(16, 2, 128, 1)))],
                     navier=[(4096, 65, True, "rbc")]),   # (a confined run would need the host eigendecomposition at 4097)
    "gen-8,4": dict(env={"B2_NOFAST": "1"},
                    spaces=[((CD, 129, CN, 257), (lay(8, 4, 16, 0), lay(8, 4, 8, 0))),
                            ((R2C, 256, CD, 129), (lay(8, 4, 8, 0), lay(8, 4, 16, 0)))],
                    navier=[(129, 129, False, "rbc")]),
    "gen-4,4": dict(env={"B2_NOFAST": "1"},
                    spaces=[((CD, 65, CN, 65), (lay(4, 4, 8, 0), lay(4, 4, 8, 0))),
                            ((R2C, 64, CDN, 65), (lay(4, 4, 8, 0), lay(4, 4, 8, 0)))],
                    navier=[(65, 65, False, "hc")]),
    "gen-16,2": dict(env={"B2_LN": "2", "B2_E": "16", "B2_NOFAST": "1"},
                     spaces=[((CD, 513, CN, 65), (lay(4, 4, 8, 0), lay(16, 2, 16, 0)))],
                     navier=[]),
    "gen-8,2": dict(env={"B2_LN": "2"},
                    spaces=[((CD, 257, CN, 257), (lay(8, 2, 16, 0), lay(8, 2, 16, 0)))],
                    navier=[(257, 257, False, "rbc")]),
    "gen-4,2": dict(env={"B2_LN": "2", "B2_E": "4"},
                    spaces=[((CD, 129, CN, 129), (lay(4, 2, 16, 0), lay(4, 2, 16, 0)))],
                    navier=[(128, 129, True, "rbc")]),
}
for _w in (2, 3, 5):   # narrow sub-chunks; 33 and 257 tiles per lane leave a partial last sub-chunk for every width
    CASES[f"chunks-{_w}"] = dict(env={"B2_CHW": str(_w)}, chw=_w,
                                 spaces=[((CD, 129, CN, 129), (lay(8, 4, 8, 1), lay(8, 4, 8, 1))),
                                         ((CD, 1025, CN, 65), (lay(4, 4, 8, 1), lay(8, 4, 64, 1)))],
                                 navier=[(129, 129, False, "rbc")] if _w == 3 else [])

# switches read once when the library loads: a child process each
FRESH_CASES = {
    "notma-generic": dict(env={"B2_NOTMA": "1", "B2_NOFAST": "1"},
                          spaces=[((CD, 129, CN, 129), (lay(8, 4, 8, 0), lay(8, 4, 8, 0)))],
                          navier=[(129, 129, False, "rbc")]),
    "ldthreads-chw3": dict(env={"B2_LDTHREADS": "1", "B2_CHW": "3"}, chw=3,
                           spaces=[((CD, 129, CN, 129), (lay(8, 4, 8, 1), lay(8, 4, 8, 1)))],
                           navier=[(129, 129, False, "rbc")]),
}
ALL_CASES = {**CASES, **FRESH_CASES}

# the layouts one GPU reaches with default settings, and the suites that check them there
DEFAULT_LAYOUTS = {
    lay(4, 4, 8, 1): "test_gpu_parity.py: 64-point lanes (65-point Chebyshev, r2c64)",
    lay(8, 4, 8, 1): "test_gpu_parity.py: 128-point lanes",
    lay(8, 4, 16, 1): "test_gpu_parity.py: 256-point lanes",
    lay(8, 4, 32, 1): "test_gpu_parity.py: 512-point lanes",
    lay(8, 4, 64, 1): "test_gpu_parity.py: 1024-point lanes",
    lay(16, 4, 64, 1): "test_gpu_parity.py, test_gpu_parity_large.py: 2048-point lanes",
    lay(16, 4, 128, 1): "test_gpu_parity.py, test_gpu_parity_large.py: 4096-point lanes",
    lay(16, 2, 256, 1): "test_gpu_parity_large.py: 8192-point lanes",
    lay(16, 4, 0, 0): "test_gpu_zz_any_size.py: lanes that are not a power of two (dense transform)",
}


def instance_of(layout):
    """the lane_kernel<E, LN, TPLC> a layout runs on: TPLC = TPL for fast layouts, 0 (generic) otherwise"""
    e, ln, tpl, fast = layout
    return (e, ln, tpl if fast else 0)


def compiled_instances():
    src = open(os.path.join(ROOT, "rustpde_mpi_b200", "csrc", "b200pde.cu")).read()
    body = src[src.index("static int launch_pass("):]
    body = body[:body.index("\n}\n")]
    fast = {tuple(int(x) for x in m) for m in re.findall(r"B2_INST\((\d+),\s*(\d+),\s*(\d+)\)", body)}
    return fast | {(e, ln, 0) for e in (16, 8, 4) for ln in (4, 2)}


def sp_name(sp):
    kind = {CH: "ch", CD: "cd", CN: "cn", CDN: "cdn", R2C: "r2c"}
    return f"{kind[sp[0]]}{sp[1]}x{kind[sp[2]]}{sp[3]}"


def max_lane(case):
    return max(max(sp[1], sp[3]) for sp, _ in case["spaces"])


# ---- the checks: run under the case's knobs (the caller sets them) ----
def space_layouts(case):
    """{space name: [layout of orient 0, layout of orient 1]} of spaces created now, plus the sub-chunk widths"""
    import rustpde_mpi_b200 as b2

    out = {}
    for sp, _ in case["spaces"]:
        s = b2.Space2((sp[0], sp[1]), (sp[2], sp[3]))
        ls = [s.lane_layout(o) for o in (0, 1)]
        out[sp_name(sp)] = {"layout": [[d["E"], d["LN"], d["TPL"], d["fast"]] for d in ls], "chw": [d["CHW"] for d in ls]}
        s.close()
    return out


def check_layouts(case, got):
    bad = []
    for sp, want in case["spaces"]:
        g = got[sp_name(sp)]
        if [tuple(x) for x in g["layout"]] != list(want):
            bad.append((sp_name(sp), g["layout"], want))
        if "chw" in case and g["chw"] != [case["chw"]] * 2:
            bad.append((sp_name(sp), "CHW", g["chw"], case["chw"]))
    return bad


def operator_errors(case):
    """{check label: relative error against the oracle} for every operator of every space of the case"""
    from tests import gpu_checks as g

    out = {}
    for sp, _ in case["spaces"]:
        name = sp_name(sp)
        out[f"{name} roundtrip_layout"] = g.check_roundtrip_layout(*sp)
        for op in ("forward", "backward", "to_ortho", "from_ortho"):
            out[f"{name} {op}"] = getattr(g, "check_" + op)(*sp)
        for d in ((1, 0), (0, 1), (2, 0), (0, 2), (1, 1)):
            out[f"{name} gradient{d}"] = g.check_gradient(*sp, d)
        if sp[0] != CH and sp[2] != CH:
            out[f"{name} hholtz_adi"] = g.check_hholtz(*sp)
        # the tensor solvers need the host eigendecomposition of a Chebyshev axis 0 (dense, so only up to 1025 points)
        if (sp[0] == R2C or (sp[0] in (CD, CN) and sp[1] <= 1025)) and sp[2] in (CD, CN):
            out[f"{name} poisson"] = g.check_poisson(*sp)
            out[f"{name} hholtz_tensor"] = g.check_hholtz_tensor(*sp)
    return out


def navier_error(nx, ny, periodic, bc):
    from tests import gpu_checks as g

    return max(g.check_navier(nx, ny, 2, periodic, bc=bc).values())


def nav_name(nv):
    nx, ny, periodic, bc = nv
    return f"navier {nx}x{ny} {'periodic' if periodic else 'confined'} {bc}"


def run_case(case):
    """layouts and errors of one case under the knobs already in the environment (JSON-ready)"""
    t0 = time.time()
    res = {"layouts": space_layouts(case), "errors": operator_errors(case)}
    for nv in case["navier"]:
        res["errors"][nav_name(nv)] = navier_error(*nv)
    res["seconds"] = time.time() - t0
    return res


def assert_case(name, case, res):
    bad_layout = check_layouts(case, res["layouts"])
    assert not bad_layout, (name, "knobs did not reach the expected layout", bad_layout)
    errs = res["errors"]
    worst = max(errs, key=errs.get)
    print(f"\n[{name}] {len(errs)} checks, largest relative error {errs[worst]:.2e} ({worst}), {res['seconds']:.1f} s")
    for k, v in errs.items():
        if k.endswith("roundtrip_layout"):
            assert v == 0.0, (name, k, v)
    bad = {k: v for k, v in errs.items() if not v < TOL}
    assert not bad, (name, bad)


# child process: python -c CHILD <emu|gpu|layouts> <case names...>; the knobs come from its environment
CHILD = r'''
import json, os, sys
sys.path.insert(0, %r)
if sys.argv[1] in ("emu", "layouts"):
    from tests import emu
    emu.activate()
from tests import test_gpu_x_lane_instances as t
out = {}
for name in sys.argv[2:]:
    case = t.ALL_CASES[name]
    if sys.argv[1] == "layouts":   # one process for every case: the layout depends on the knobs at space creation only
        for k in t.KNOBS:
            os.environ.pop(k, None)
        os.environ.update(case["env"])
        out[name] = t.space_layouts(case)
    else:
        out[name] = t.run_case(case)
print("RESULT " + json.dumps(out))
''' % ROOT


def run_child(mode, names, env, timeout):
    base = {k: v for k, v in os.environ.items() if k not in KNOBS}
    r = subprocess.run([sys.executable, "-c", CHILD, mode, *names], capture_output=True, text=True, timeout=timeout, cwd=ROOT,
                       env=dict(base, **env))
    lines = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert r.returncode == 0 and lines, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(lines[-1][len("RESULT "):])


# ---- on the GPU ----
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_lane_instance(name, monkeypatch):
    case = CASES[name]
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)
    assert_case(name, case, run_case(case))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FRESH_CASES))
def test_lane_load_switches(name):
    case = FRESH_CASES[name]
    res = run_child("gpu", [name], case["env"], timeout=900)[name]
    assert_case(name, case, res)


# ---- on the CPU ----
def test_layout_table_covers_every_instance():
    """Each case's knobs reach the layout the table expects, and the cases together with the default layouts reach every
    compiled lane_kernel instance -- a new instance fails this test until a case runs it."""
    got = run_child("layouts", list(ALL_CASES), {}, timeout=900)
    bad = {name: check_layouts(case, got[name]) for name, case in ALL_CASES.items()}
    assert not any(bad.values()), {k: v for k, v in bad.items() if v}
    reached = {instance_of(l) for case in ALL_CASES.values() for _, ls in case["spaces"] for l in ls}
    reached |= {instance_of(l) for l in DEFAULT_LAYOUTS}
    assert reached == compiled_instances(), (sorted(compiled_instances() - reached), sorted(reached - compiled_instances()))
    assert len(compiled_instances()) == 20


EMU_CASES = [n for n, c in ALL_CASES.items() if max_lane(c) <= 1025 and all(max(nv[:2]) <= 1025 for nv in c["navier"])]


@pytest.mark.parametrize("name", EMU_CASES)
def test_emulated_instance_table(name):
    """The same checks on the same sources in the CPU SIMT emulator (host logic only: says nothing about GPU results)."""
    case = ALL_CASES[name]
    assert_case(name, case, run_child("emu", [name], case["env"], timeout=1800)[name])
