"""The pixel observation's configuration without a GPU: cfg.pixel_obs in the C ABI, the sizes agarcl_make_layout accepts and
the combinations it refuses, snapshot slots that do not depend on it, and k_draw_views compiled without spills."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import pytest

from agarcl_b200 import make_cfg
from agarcl_b200._lib import AgarclError, make_layout, snapshot_slot_bytes


def test_pixel_obs_is_the_last_field_of_the_cfg():
    from agarcl_b200._abi import Cfg
    c = make_cfg(pixel_obs=96)
    assert C.sizeof(Cfg) == 28 * 4 and c.pixel_obs == 96
    assert C.c_int32.from_buffer(c, 27 * 4).value == 96
    c.pixel_obs = 0
    assert bytes(c)[27 * 4:] == b"\0\0\0\0"


@pytest.mark.parametrize("S", [16, 48, 64, 128, 144, 256, 1024, 2048])
def test_accepted_sizes(S):
    plain = make_layout(make_cfg())
    assert bytes(make_layout(make_cfg(pixel_obs=S))) == bytes(plain)
    make_layout(make_cfg(pixel_obs=S, ram_obs=1))


@pytest.mark.parametrize("kw,text", [
    (dict(pixel_obs=8), "multiple of 16"), (dict(pixel_obs=24), "multiple of 16"), (dict(pixel_obs=2064), "multiple of 16"),
    (dict(pixel_obs=4096), "multiple of 16"), (dict(pixel_obs=-16), "multiple of 16"),
    (dict(pixel_obs=64, num_frames=2), "num_frames"), (dict(pixel_obs=64, num_frames=4), "num_frames"),
    (dict(pixel_obs=64, strict_reference=1), "strict_reference"), (dict(pixel_obs=64, ram_obs=2), "ram_obs = 2")])
def test_refused_configurations(kw, text):
    with pytest.raises(AgarclError, match=text):
        make_layout(make_cfg(**kw))


@pytest.mark.parametrize("kw", [dict(), dict(ram_obs=1), dict(num_agents=4, mode_number=5, num_bots=0)])
def test_snapshot_slots_do_not_depend_on_pixels(kw):
    assert snapshot_slot_bytes(make_cfg(pixel_obs=128, **kw)) == snapshot_slot_bytes(make_cfg(**kw))


def test_draw_kernels_have_no_spills():
    from agarcl_b200 import build
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, "draw_kernel.cu"), "-o", os.path.join(d, "k.o")],
                           capture_output=True, text=True, check=True)
    text = r.stdout + r.stderr
    blocks = re.findall(r"Function properties for (\S*k_draw\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill "
                        r"loads", text)
    assert sorted(n for n, *_ in blocks) == ["_ZN2ag12k_draw_viewsENS_10DrawParamsE", "_ZN2ag6k_drawENS_10DrawParamsE"], text
    for name, stack, st, ld in blocks:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), (name, stack, st, ld)
