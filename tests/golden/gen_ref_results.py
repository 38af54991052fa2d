"""Records into tests/golden/ref_results/ the answers of the unmodified reference
runtime that the tests compare against, so that the comparisons also run where
oracle/_ref cannot be built (oracle/ref.py replays them there, keyed by a digest
of each call's inputs).  Needs oracle/_ref: `make -C oracle/ref REF=<reference
source tree>`, or build() with HS_REFERENCE set.

  python tests/golden/gen_ref_results.py          CPU tests, and the device tests on the SIMT emulator
  python tests/golden/gen_ref_results.py --gpu    the device tests on a CUDA device (the emulator skips some)

Answers already in the store are kept and, where the runtime is built, every
test run checks them against it.  After a change to what the compiler emits,
delete the store and run both commands again."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def run(extra_env, args):
    env = dict(os.environ, HS_REF_RECORD="1", **extra_env)
    subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider"] + args, cwd=ROOT, env=env,
                   check=True)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    import oracle.ref as ref
    if not ref.live():
        raise SystemExit("oracle/_ref is not built: nothing to record")
    if "--gpu" in sys.argv:
        run({}, ["-m", "gpu", "tests"])
    else:
        run({}, ["-m", "not gpu", "tests"])
        run({"HSB200_EMU": "1"}, ["-m", "gpu", "tests"])
