"""The kernels' device functions (hexb_core.cuh, hexb_phases.cuh, hexb_views.cuh, hexb_search.cuh, hexb_mcts.cuh) under
AddressSanitizer and UndefinedBehaviorSanitizer: the host emulator (tests/emu/hexb_emu.cpp) is built with -fsanitize=address,undefined
and the emulator parity tests are run against that build (compute-sanitizer is closed on this GPU pool, so this is the memory / UB
check the device LOGIC gets; races between lanes are not modelled - the emulator replays the lanes serially).

Usage: python tools/emu_sanitize.py [pytest -k expression]     exit code = pytest's"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build(out_dir=None):
    """The sanitizer build of the emulator, kept beside the ordinary one (git-ignored) and rebuilt when a source is newer."""
    out_dir = out_dir or os.path.join(ROOT, "tests", "emu")
    so = os.path.join(out_dir, "libhexb_emu_san.so")
    srcs = [os.path.join(ROOT, "tests", "emu", "hexb_emu.cpp")] + [
        os.path.join(ROOT, "hex_gym_env_b200", "csrc", f)
        for f in ("hexb_core.cuh", "hexb_phases.cuh", "hexb_views.cuh", "hexb_search.cuh", "hexb_mcts.cuh")]
    asan = subprocess.run(["g++", "-print-file-name=libasan.so"], stdout=subprocess.PIPE, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        return None, "libasan.so not found"
    if os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(x) for x in srcs):
        return so, asan
    cmd = ["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-Wno-unknown-pragmas", "-fsanitize=address,undefined",
           "-fno-sanitize-recover=undefined", "-o", so, srcs[0]]
    cc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if cc.returncode != 0:
        return None, cc.stdout
    return so, asan


def run(select=None, extra=()):
    so, asan = build()
    if so is None:
        return None, asan
    env = dict(os.environ, HEXB_EMU_LIB=so, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0", UBSAN_OPTIONS="print_stacktrace=1")
    cmd = [sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_emu_parity.py"), "-x", "-q", "-p", "no:cacheprovider",
           "--deselect", "tests/test_emu_parity.py::test_device_logic_under_address_and_ub_sanitizers"]
    if select:
        cmd += ["-k", select]
    out = subprocess.run(cmd + list(extra), env=env, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return out.returncode, out.stdout


if __name__ == "__main__":
    rc, text = run(sys.argv[1] if len(sys.argv) > 1 else None)
    print(text[-4000:])
    sys.exit(2 if rc is None else rc)
