"""CPU: conflux::conflux_layout of this repo's facade is field-for-field identical to the COSTA descriptors the
REFERENCE's conflux_layout / lu_params::matrix produce (layout.cpp:30-135), for both overloads, both orderings, several
grids.  The reference side is stored in tests/golden/layouts.txt (tests/golden/make_golden.py layouts); the facade side
is compiled here (tests/cpp/layout_dump.cpp) and answers the same cases in the same format."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_layout_descriptors_match_costa(tmp_path, golden_dir):
    exe = tmp_path / "layout_dump"
    subprocess.check_call(["g++", "-O1", "-std=c++17", f"-I{ROOT}/include", f"{ROOT}/tests/cpp/layout_dump.cpp", "-o", str(exe)])
    golden = open(os.path.join(golden_dir, "layouts.txt")).read().splitlines()
    cases = [ln for ln in golden if ln.startswith("case ")]
    assert len(cases) == 63
    out = subprocess.run([str(exe)], input="\n".join(cases) + "\n", capture_output=True, text=True, check=True)
    mine = out.stdout.splitlines()
    case = None
    for a, b in zip(mine, golden):
        case = a if a.startswith("case ") else case
        assert a == b, f"{case}: {a!r} != reference {b!r}"
    assert len(mine) == len(golden)
