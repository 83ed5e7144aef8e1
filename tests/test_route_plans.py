"""Host-side checks of the round-2 route planners (no GPU): tools/route_plan_dump.cu is compiled with nvcc and run here.
K2 (persistent tcgen05 1x1 conv) plans of the late expands / gated projects / head conv, KD (depthwise + squeeze) chunk widths,
thread counts and shared memory, pw_tc3's walk over the tiles of the early gated projects."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMEM_OPTIN = 227 * 1024          # dynamic + static shared memory one CTA may use on sm_100


@pytest.fixture(scope="module")
def dump(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("plans") / "route_plan_dump")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    r = subprocess.run([nvcc, "-std=c++17", "-arch=sm_100a", "-o", exe, os.path.join(ROOT, "tools", "route_plan_dump.cu")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr

    def run(crops):
        out = subprocess.run([exe, str(crops)], capture_output=True, text=True, check=True).stdout
        kd, k2, pw3 = {}, {}, {}
        for line in out.splitlines():
            m = re.search(r"kd b(\d+) cc (\d+) threads (\d+) strips (\d+) pw (\d+) smem (\d+) chunks (\d+)", line)
            if m:
                kd[int(m.group(1))] = dict(zip("cc threads strips pw smem chunks".split(), (int(v) for v in m.groups()[1:])))
            m = re.search(r"k2 (\w+)\s+b(\d+) M (\d+) K (\d+) N (\d+) gate (\d) : n_tile (\d+) n_tiles (\d+) tiles (\d+) nkb (\d+) stages (\d+) "
                          r"resident (\d) tmem (\d+) smem (\d+)", line)
            if m:
                k2[(m.group(1), int(m.group(2)))] = dict(zip("M K N gate n_tile n_tiles tiles nkb stages resident tmem smem".split(),
                                                             (int(v) for v in m.groups()[2:])))
            m = re.search(r"pw3 b(\d+) tiles_per_crop (\d+) tpc (\d+) groups (\d+) umma_n (\d+) tmem (\d+) smem (\d+)", line)
            if m:
                pw3[int(m.group(1))] = dict(zip("tiles_per_crop tpc groups umma_n tmem smem".split(), (int(v) for v in m.groups()[1:])))
            if "not taken" in line:
                pw3[int(re.search(r"b(\d+)", line).group(1))] = None
        return kd, k2, pw3
    return run


def test_kd_instances(dump):
    kd, _, _ = dump(256)
    assert sorted(kd) == [1, 7, 9, 10, 12, 13, 16]                 # one line per distinct late-block shape + block 1
    cexp = {1: 32, 7: 480, 9: 480, 10: 672, 12: 672, 13: 1152, 16: 1152}
    for b, r in kd.items():
        assert cexp[b] % r["cc"] == 0 and r["chunks"] == cexp[b] // r["cc"]
        assert r["threads"] % 32 == 0 and r["strips"] * (r["cc"] // 4) <= r["threads"] < r["strips"] * (r["cc"] // 4) + 32
        assert r["smem"] + 1024 <= SMEM_OPTIN
        assert (r["pw"] * r["pw"] * r["cc"] * 2) % 16 == 0        # the tile box is a whole number of 16-byte TMA units
    # the 14x14 / 3x3 instances keep four CTAs per SM, the 5x5 ones three
    assert kd[7]["smem"] * 4 <= 228 * 1024 and kd[10]["smem"] * 3 <= 228 * 1024
    assert kd[1]["pw"] == 16 and kd[9]["pw"] == 18 and kd[12]["pw"] == 17 and kd[13]["pw"] == 11 and kd[16]["pw"] == 9


def test_k2_plans(dump):
    _, k2, _ = dump(256)
    for key, r in k2.items():
        assert r["smem"] <= 225 * 1024, key                       # launch_k2 opts in to 225 KB
        assert r["tmem"] in (32, 64, 128, 256, 512) and 2 * r["n_tile"] <= r["tmem"], key       # two accumulators
        assert r["n_tile"] % 16 == 0 and r["n_tile"] <= 256 and r["n_tile"] * r["n_tiles"] >= r["N"], key
        assert r["nkb"] == (r["K"] + 63) // 64 and 2 <= r["stages"] <= 8, key
        assert r["tiles"] == ((r["M"] + 127) // 128) * r["n_tiles"], key
        if r["resident"]:
            assert r["n_tiles"] == 1 and r["stages"] >= 3, key    # weights stay only next to a ring of three A stages or more
    # the projects up to block 11 keep their weights resident (82 / 115 / 154 KB), the 7x7 ones (270+ KB) stream them
    assert k2[("project", 7)]["resident"] and k2[("project", 9)]["resident"] and k2[("project", 10)]["resident"]
    assert not k2[("project", 12)]["resident"] and not k2[("project", 13)]["resident"] and not k2[("project", 16)]["resident"]
    # expands: fp16 output, several n tiles, never resident
    assert all(not r["resident"] for (kind, _), r in k2.items() if kind == "expand")
    # launch_pw sends a conv to K2 only when it has at least 2 x 148 tiles: at 256 crops per stream that is every expand and
    # the 14x14 projects; the 7x7 projects (98 / 196 tiles) and every small batch stay on pw_tc2
    assert min(r["tiles"] for (kind, _), r in k2.items() if kind == "expand") >= 296
    assert k2[("project", 10)]["tiles"] >= 296 > k2[("project", 13)]["tiles"]
    _, small, _ = dump(8)
    assert max(r["tiles"] for r in small.values()) < 296


def test_pw_tc3_rule(dump):
    _, _, pw3 = dump(256)
    assert pw3[1] is not None and all(pw3[b] is None for b in (2, 3, 4, 5, 6))        # K <= 64 only: block 1
    r = pw3[1]
    assert r["tiles_per_crop"] == 98 and r["tpc"] >= 3 and r["tpc"] * r["groups"] >= 98 > r["tpc"] * (r["groups"] - 1)
    assert r["umma_n"] == 16 and r["tmem"] == 32 and r["smem"] <= 200 * 1024
    # small batches: too few tiles per CTA to pipeline -> pw_tc2 (bit-identical, so the switch is invisible)
    _, _, small = dump(8)
    assert small[1] is None
    _, _, mid = dump(70)
    assert mid[1] is not None and mid[1]["tpc"] == 5 and mid[1]["groups"] == 20
