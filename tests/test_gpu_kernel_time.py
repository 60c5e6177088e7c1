"""cucd_last_kernel_time after host-buffer batch calls: a call that goes through the device staging blocks is timed; a call small
enough for the zero-copy path (its kernels read and write page-locked host memory) is not, and the query then fails instead of
returning the time of an earlier call."""
import os

import numpy as np
import pytest

from _util import all_cus, pseudo_recon, textured_plane

pytestmark = pytest.mark.gpu

W = H = 512
M = 64
# the small calls move well under 4 KB; the large ones more than 1 MB each way or back, which always takes the staged path
SMALL_DIRECT = int(os.environ.get("CUCD_DIRECT_LIMIT", 96 << 10)) >= 4096


def tu_call(eng, rng, small):
    n_tu, log2 = (1, 3) if small else (256, 5)
    n = 1 << log2
    org = rng.integers(0, 256, n_tu * n * n).astype(np.int16)
    border = rng.integers(0, 256, n_tu * (4 * n + 1)).astype(np.int16)
    eng.intra_tu_code([(log2, int(m), 32, 0) for m in rng.integers(0, 35, n_tu)], org, border)


def tmv_call(eng, rng, small):
    cus = all_cus(W, H, depths=(1, 2, 3))
    eng.tmv_features(cus[:1] if small else cus)


def me_call(eng, rng, small):
    if small:
        descs = [dict(x=64, y=64, w=8, h=8, ref_idx=0, left=-4, right=4, top=-4, bottom=4, sub_shift=0)]
    else:
        descs = [dict(x=int(x), y=int(y), w=16, h=16, ref_idx=0, left=-32, right=32, top=-32, bottom=32, sub_shift=1)
                 for x, y in zip(rng.integers(0, 31, 128) * 16, rng.integers(0, 31, 128) * 16)]
    eng.me_sad_surface(descs)


@pytest.mark.parametrize("small", [False, True], ids=["staged", "zero_copy"])
@pytest.mark.parametrize("call", [tu_call, tmv_call, me_call], ids=["tu", "tmv", "me"])
def test_last_kernel_time_after_call(cucd, call, small):
    rng = np.random.default_rng(11)
    org = textured_plane(W, H, 8, seed=11)
    with cucd.Engine(W, H, bit_depth=8) as eng:
        eng.set_cur_picture(org)
        eng.set_ref_picture(0, np.pad(pseudo_recon(org, 8), M, mode="edge"), M, M)
        call(eng, rng, small=False)
        assert eng.last_kernel_time_ms() > 0
        if not small:
            return
        call(eng, rng, small=True)                      # after a timed call: the query must not report that call's time
        if SMALL_DIRECT:
            with pytest.raises(cucd.CucdError, match="was not timed"):
                eng.last_kernel_time_ms()
        else:
            assert eng.last_kernel_time_ms() > 0
