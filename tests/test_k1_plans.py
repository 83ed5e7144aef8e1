"""Host-side checks of the K1 tile planner (no GPU): tools/k1_plan_dump.cu is compiled with nvcc and run here."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LINE = re.compile(r"b(\d+)\s+(\d+)->\s*(\d+) k(\d) s(\d) cin\s*(\d+) cexp\s*(\d+) :\s*(\d+)x(\d+)\s+r(\d) cc(\d+)\s+nt(\d+) nb(\d)\s+mtiles (\d) "
                  r"rows_alloc\s+(\d+) tmem\s+(\d+) chunks\s+(\d+) PY\s+(\d+) PYc\s+(\d+) smem\s+(\d+) \(A\s+(\d+) W\s+(\d+) C\s+(\d+) E\s+(\d+)\) (\d)/SM")
KEYS = "idx hin ho k s cin cexp th tw r cc nt nb mtiles rows_alloc tmem chunks PY PYc smem A W C E per_sm".split()


@pytest.fixture(scope="module")
def dump(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("plans") / "k1_plan_dump")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    r = subprocess.run([nvcc, "-std=c++17", "-arch=sm_100a", "-o", exe, os.path.join(ROOT, "tools", "k1_plan_dump.cu")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr

    def run(*plan):
        out = subprocess.run([exe] + [str(v) for v in plan], capture_output=True, text=True, check=True).stdout
        rows = []
        for line in out.splitlines():
            m = LINE.search(line)
            if m:
                d = dict(zip(KEYS, (int(v) for v in m.groups())))
                d["alt"] = line.lstrip().startswith("alt")
                rows.append(d)
        return rows
    return run


def test_every_block_has_a_plan_that_fits(dump):
    rows = [r for r in dump() if not r["alt"]]
    assert [r["idx"] for r in rows] == [2, 3, 4, 5, 6, 7, 9, 10, 12, 13, 16]      # one line per distinct block shape
    for r in rows:
        assert r["smem"] <= 227 * 1024 - 256
        assert r["cexp"] % r["cc"] == 0 and r["cc"] % 16 == 0
        assert r["mtiles"] * r["cc"] <= r["tmem"] <= 512 and r["tmem"] & (r["tmem"] - 1) == 0
        assert r["rows_alloc"] % 8 == 0 and r["rows_alloc"] <= r["mtiles"] * 128
        assert r["PY"] == r["PYc"] * r["nb"] and r["PY"] * (r["cc"] // 4) <= r["nt"]
        assert r["nb"] * r["cc"] <= r["nt"]                         # one thread per (crop, channel) in the squeeze reduction
        two = r["nt"] == 256 and r["smem"] <= 115000 and r["tmem"] <= 256
        assert r["per_sm"] == (2 if two else 1)
    by = {r["idx"]: r for r in rows}
    # the GEMM rows are the halo pixels inside the image: 14x14 inputs with a 5x5 window need 196 rows, not 18*18
    assert by[10]["rows_alloc"] == 200 and by[10]["mtiles"] == 2
    assert by[12]["rows_alloc"] == 200                            # stride 2: the whole 14x14 input of a 7x7 output tile
    # 7x7 stages: two crops share one M tile (2 * 49 rows)
    assert by[13]["nb"] == 2 and by[13]["rows_alloc"] == 104 and by[13]["mtiles"] == 1
    # early blocks keep two CTAs per SM
    for i in (2, 3, 4, 5, 6):
        assert by[i]["per_sm"] == 2, by[i]


def test_candidate_rules(dump):
    # two crops per CTA only where one tile is the whole image
    alts = [r for r in dump(7, 7, 4, 48, 256, 2) if r["alt"]]
    assert {r["idx"] for r in alts} == {13, 16}
    # an interior 8x8 stride-2 tile has 17x17 halo pixels (3 M tiles); 8x7 fits two
    alts = {r["idx"]: r for r in dump(8, 7, 4, 48, 256, 1) if r["alt"]}
    assert alts[2]["rows_alloc"] == 256 and alts[2]["mtiles"] == 2
    # shapes that do not divide the output are refused
    assert not [r for r in dump(5, 5, 4, 48, 256, 1) if r["alt"]]
