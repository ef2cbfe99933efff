"""Kernel variants that are selected through the environment when the library first launches them (A/B switches kept for
measurement: FYX_CULL_VARIANT, FYX_SKIN_VARIANT) get the same bit-exact parity tests as the defaults, each in its own
process."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _run(env, tests, k):
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-k", k] + [os.path.join(HERE, t) for t in tests],
                       capture_output=True, text=True, env=e, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


@pytest.mark.timeout(1000)
@pytest.mark.parametrize("variant", ["0", "3", "13", "20", "34", "52"])
def test_cull_variants_match_the_oracle(variant):
    """bit 0: warp-union pre-reject of whole frusta, bit 1: warp-wide compaction, bit 2: FYX_UPDATE_ALL specialisation, bit 3: deferred compaction (k_compact_vis), bit 4: 32-register build, bit 5: warp-convergent predicate
    (fyx_kernels.cu; the default is 20).  Four variants exercise every bit; the others differ only in combinations."""
    _run({"FYX_CULL_VARIANT": variant}, ["test_gpu_parity.py", "test_gpu_drawprep.py", "test_gpu_shapes.py"],
         "cull or render_prep or pipelined or k7 or lod or light or instances or bundle")


@pytest.mark.timeout(1000)
@pytest.mark.parametrize("variant", ["tma2", "tma3", "pair4", "pair5", "pair6"])  # TMA rings (2 / 3 stages); two vertices per thread, 4 / 5 / 6 CTAs per SM
def test_tma_skinning_variants_match_the_oracle(variant):
    """k_skin_tma: vertex blocks staged by cp.async.bulk + mbarrier rings; k_skin2: two vertices per thread (fyx_kernels.cu)."""
    _run({"FYX_SKIN_VARIANT": variant}, ["test_gpu_parity.py", "test_gpu_fullsize.py", "test_gpu_shapes.py"], "skin or render_prep")


@pytest.mark.timeout(1000)
@pytest.mark.parametrize("mode", ["0", "1"])
def test_subforest_kernel_on_and_off_match_the_oracle(mode):
    """FYX_SUBFOREST: the deep levels of the hierarchy in one launch (k_update_subforest) or one launch per level — forced
    both ways over the hierarchy / cull / skinning / animation parity tests (the default picks by level width: on for most
    of the small test scenes, so "1" mostly adds the wide ones)."""
    _run({"FYX_SUBFOREST": mode}, ["test_gpu_parity.py", "test_gpu_anim.py", "test_gpu_drawprep.py", "test_gpu_shapes.py"], "not cpp_host and not k6 and not k7")


@pytest.mark.timeout(1000)
def test_fold_in_stream_order_matches_the_oracle():
    """FYX_SIDE_FOLD=0: asynchronous frames run the skinned-mesh fold in order on the main stream instead of beside the palette /
    skinning kernels (the default, exercised by every pipelined test of the normal run)."""
    _run({"FYX_SIDE_FOLD": "0"}, ["test_gpu_parity.py", "test_gpu_fuzz.py", "test_gpu_shapes.py"], "pipelined or render_prep or random_call or skin")
