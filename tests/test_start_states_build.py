"""Start states without a GPU: k_start_states compiles for sm_100a without stack or spills beside k_snapshot's two
directions."""
import os
import re
import subprocess
import tempfile


def test_k_start_states_has_no_spills():
    from agarcl_b200 import build
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, "snapshot_kernel.cu"),
                                             "-o", os.path.join(d, "snapshot_kernel.o")], capture_output=True, text=True, check=True)
    text = r.stdout + r.stderr
    blocks = re.findall(r"Function properties for (\S*k_start_states\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads", text)
    assert len(blocks) == 1, text
    assert tuple(int(x) for x in blocks[0][1:]) == (0, 0, 0), blocks
