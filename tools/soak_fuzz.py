"""One-off soak on a GPU box: hundreds of seeds of tests/parity.py::api_fuzz (random walks over the step / reset API against the
oracle) through the C ABI, each with a launch form (1 / 4 warps per chunk, or the library's choice) and an observation
dtype picked from the seed. python tools/soak_fuzz.py [first_seed] [count]"""
import sys, os
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import parity
from gpu_adapter import make_with
bad = 0
first = int(sys.argv[1]) if len(sys.argv) > 1 else 100
count = int(sys.argv[2]) if len(sys.argv) > 2 else 600
for seed in range(first, first + count):
    form = (0, 1, 4)[seed % 3]
    f32 = (seed // 3) % 3 == 0
    try:
        parity.api_fuzz(make_with(launch_form=form, obs_f32=f32), seed, T=40)
    except AssertionError as e:
        bad += 1
        print("FAIL", seed, form, f32, str(e)[:200])
print("soak done: %d seeds, failures: %d" % (count, bad))
