"""The cell archive without a GPU: the archive kernels compile for sm_100a without stack or spills."""
import os
import re
import subprocess
import tempfile

KERNELS = ("k_archive_cells", "k_archive_commit", "k_archive_select", "k_archive_base")


def test_archive_kernels_have_no_spills():
    from agarcl_b200 import build
    assert "archive_kernel.cu" in build.SOURCES
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, "archive_kernel.cu"),
                                             "-o", os.path.join(d, "archive_kernel.o")], capture_output=True, text=True, check=True)
    text = r.stdout + r.stderr
    blocks = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                        text)
    found = {k: tuple(int(x) for x in rest) for name, *rest in blocks for k in KERNELS if k in name}
    assert set(found) == set(KERNELS), text
    assert all(v == (0, 0, 0) for v in found.values()), found
