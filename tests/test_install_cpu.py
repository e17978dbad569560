"""CPU: a non-editable install of the package is self-contained - it carries the C ABI header (hex_gym_env_b200/include/hexb.h,
kept identical to the repository's canonical include/hexb.h), every source the library is built from, and a prebuilt library
loads from it with every declared symbol."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_packaged_header_is_the_canonical_one():
    a = open(os.path.join(ROOT, "include", "hexb.h"), "rb").read()
    b = open(os.path.join(ROOT, "hex_gym_env_b200", "include", "hexb.h"), "rb").read()
    assert a == b, "hex_gym_env_b200/include/hexb.h differs from include/hexb.h (hex_gym_env_b200._native.build() syncs them)"


def test_pip_install_target_is_self_contained(tmp_path):
    target = tmp_path / "site"
    work = tmp_path / "src"          # build from a copy: setuptools writes build/ and *.egg-info next to pyproject.toml
    lib = os.path.join(ROOT, "hex_gym_env_b200", "libhexb.so")
    if not os.path.exists(lib):
        pytest.skip("libhexb.so has not been built in this tree")
    # the package's current sources (the tree need not be a git checkout), without the products of an in-tree build
    shutil.copytree(os.path.join(ROOT, "hex_gym_env_b200"), str(work / "hex_gym_env_b200"),
                    ignore=shutil.ignore_patterns("build", "__pycache__", "*.so", "*.lock", "*.tmp"))
    shutil.copy(os.path.join(ROOT, "pyproject.toml"), str(work))
    shutil.copy2(lib, str(work / "hex_gym_env_b200" / "libhexb.so"))   # the prebuilt library ships with the package
    os.utime(str(work / "hex_gym_env_b200" / "libhexb.so"))     # the library is newer than its sources: the install must not rebuild
    r = subprocess.run([sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps", "--quiet",
                        "--target", str(target), str(work)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]
    pkg = target / "hex_gym_env_b200"
    assert (pkg / "include" / "hexb.h").is_file() and (pkg / "csrc" / "hexb_step.cuh").is_file() and (pkg / "csrc" / "hexb_host.h").is_file()
    assert (pkg / "libhexb.so").is_file()
    code = ("import ctypes, os, hex_gym_env_b200\n"
            "from hex_gym_env_b200 import _native\n"
            "assert os.path.dirname(_native.__file__).startswith(%r), _native.__file__\n"
            "assert all(os.path.exists(s) for s in _native.SOURCES), [s for s in _native.SOURCES if not os.path.exists(s)]\n"
            "L = _native.lib()\n"       # loads the installed library: no rebuild, no FileNotFoundError on a missing header
            "assert all(hasattr(L, n) for n in _native.SYMBOLS)\n"
            "print('ok', L.hexb_version())\n" % str(target))
    env = dict(os.environ, PYTHONPATH=str(target))
    r = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-3000:]
