"""Generate tests/golden/reference_bench_calls.json: the calls the reference's UNMODIFIED acceptance harness
(bench/bench.py of a checkout of the reference) makes into the engine, recorded while it drives ssd_b200 through the
`ssd` compat shim on CPU (device runner doubled, as in tests/test_reference_harness_cpu.py, which replays them).

    python oracle/gen_harness_golden.py <reference checkout>
"""
import json
import os
import runpy
import sys
import tempfile
from pathlib import Path

import pytest

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))

from tests import test_reference_harness_cpu as T  # noqa: E402

RUNS = {
    "spec": ["--size", "8", "--spec", "--k", "6", "--random", "--numseqs", "5", "--input_len", "40", "--output_len", "60",
             "--b", "2"],
    "sweep": ["--size", "8", "--random", "--numseqs", "3", "--input_len", "16", "--output_len", "20", "--b", "2",
              "--sweep", json.dumps([{"b": 2, "temp": 0.5}, {"b": 1}])],
}


def record(ref: str, argv: list[str]) -> dict:
    with pytest.MonkeyPatch.context() as mp, tempfile.TemporaryDirectory() as tmp:
        T.engine_env(Path(tmp), mp)
        calls, _ = T.spy_engine(mp, tmp)
        for mod in ("bench_helpers", "bench_paths"):  # they bind SSD_HF_CACHE at import time
            mp.delitem(sys.modules, mod, raising=False)
        mp.setattr(sys, "argv", ["bench.py"] + argv)
        mp.syspath_prepend(os.path.join(ref, "bench"))
        try:
            runpy.run_path(os.path.join(ref, "bench", "bench.py"), run_name="__main__")
        except SystemExit as ex:
            assert ex.code == 0, f"reference bench.py exited with {ex.code}"
    return {"argv": argv, **calls}


def main():
    ref = sys.argv[1]
    out = {name: record(ref, argv) for name, argv in RUNS.items()}
    path = REPO / "tests" / "golden" / "reference_bench_calls.json"
    path.write_text(json.dumps(out, indent=None, separators=(",", ":")) + "\n")
    print(path, path.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
