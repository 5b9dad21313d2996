"""CPU suite: the scan-plan scenes of tests/scan_scenes.py land on the arms they are meant to test.

tests/test_scan_plans_gpu.py compares every arm of the F32 hit scan with the oracle on these scenes.  That only tests what it
claims if each scene really selects the arm listed for it, so the numpy mirror of the host rules (scan_scenes.scan_arm) is
checked here against the numbers the rules are written in, and the matrix must reach all five arms.
"""
import pytest

import scan_scenes as ss
from rtiow_b200.capi import F64, SCAN_AUTO, SCAN_FP32, SCAN_TENSOR


def test_constants_read_from_the_headers():
    assert (ss.CAND_CAP, ss.UMMA_GROUPS, ss.UMMA_CHUNK) == (16, 6, 64)
    # the sizes where the rules flip, restated from the byte counts: npad 3200 is the largest tensor image in 227 KB, np 3040
    # the largest FP32 table beside 256 lists in 56 KB, np 13472 the largest beside 512 lists in 227 KB
    assert ss.umma_smem_bytes(3200) <= ss.SMEM_CTA < ss.umma_smem_bytes(3264)
    assert (4 * 3040 + 16) * 4 + 256 * 32 <= ss.SMEM_SMALL < (4 * 3072 + 16) * 4 + 256 * 32
    assert (4 * 13472 + 16) * 4 + 512 * 32 <= ss.SMEM_CTA < (4 * 13504 + 16) * 4 + 512 * 32


@pytest.mark.parametrize("name", sorted(ss.SCENES))
def test_scene_lands_in_its_arm(capi, name):
    arrays = ss.build(name, capi)
    want = ss.SCENES[name][1]
    for backend in (SCAN_AUTO, SCAN_FP32, SCAN_TENSOR):
        assert ss.scan_arm(arrays, backend)[0] == want[backend], (name, backend)
    assert ss.scan_arm(arrays, SCAN_AUTO, precision=F64)[0] == "F64"


def test_each_rule_fails_alone_at_its_boundary(capi):
    """one scene per rule that can fail, failing that rule and no other; and the scenes just inside each rule"""
    info = {name: ss.scene_info(ss.build(name, capi)) for name in ss.SCENES if not name.startswith("compact-13")}
    assert info["compact-3201"]["failing"] == ["smem"] and info["compact-3201"]["npad"] == 3264
    assert info["compact-3200"]["failing"] == [] and info["compact-3137"]["npad"] == 3200 and info["compact-3137"]["failing"] == []
    assert info["row-r0.2"]["failing"] == ["slack"]
    assert info["row-r0.4"]["failing"] == [] and info["row-r0.4"]["slack"] > 0.95 * info["row-r0.4"]["mean_r2"]
    assert info["ball-R130"]["failing"] == ["d_fits"]
    r121 = info["ball-R121"]
    assert r121["failing"] == [] and r121["Rp"] == 128 and 1 <= r121["ns"] % 64 <= 32 and r121["np"] < r121["npad"]
    # the scenes that straddle the FP32 segment of 1024 spheres and its partial last word
    for name, words, tail in (("compact-1031", 32, 2), ("compact-1057", 33, 1), ("compact-1100", 34, 3)):
        n_rec = -(-info[name]["ns"] // 4)
        assert (n_rec >> 3, n_rec & 7) == (words, tail), name
    assert all(info[f"compact-{n}"]["failing"] == [] for n in (1, 63, 64, 65, 127, 129, 1031))


def test_the_matrix_covers_every_arm():
    arms = {arm for _, want in ss.SCENES.values() for arm in want.values()} | {"F64"}
    assert arms - {None} == set(ss.ARMS)
