"""tools/sass_footprint.py names the rollout_kernel flavours by their mangled names; every one must exist in the objects
build.py leaves (CPU only: the library is built for sm_100a without a GPU and the objects are read with cuobjdump)."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_footprint_kernel_is_in_its_object():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_footprint as sf
    from neuro_genetic_pong_self_play_b200 import build
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("needs the CUDA toolkit's cuobjdump")
    build.build()
    sections = {}
    for key, name in sf.KERNELS.items():
        obj = sf.default_object(key)
        if obj not in sections:
            sections[obj] = subprocess.run([cuobjdump, "-elf", obj], check=True, capture_output=True, text=True).stdout
        assert f".text.{name}" in sections[obj], (key, name, obj)
