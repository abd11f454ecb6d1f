"""Which kernel instantiations of libgenpc_b200.so does the GPU suite launch?

    python tools/kernel_coverage.py [--json PATH] [pytest args ...]      (default: every tests/test_*.py with -m gpu -q)

Runs pytest with a plugin that wraps the call phase of every test in torch.profiler (CUDA activity) and records the kernels
it launched.  By default each test file runs in a child process of its own, pytest in-process there: after a few hundred
profiling sessions in one process the profiler was seen to return traces without kernels for short windows.  Tests that
profile their own calls (a module-level `launched_kernels` helper, as in tests/test_dispatch_paths.py) are not wrapped --
profilers do not nest -- and what their helper sees is recorded instead.
Prints, for every instantiation in the library (cuobjdump -sass), whether a test launched it and its entry in
tests/test_kernel_inventory.py; the list of instantiations that no test launched comes last.  Kernels launched in child
processes (the C API test, the two-rank NCCL worker) are not seen.  --json writes {kernel: [test ids]}."""
import json
import os
import subprocess
import sys
import tempfile
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pytest  # noqa: E402

from test_kernel_inventory import KERNELS, kernel_key, library_kernels  # noqa: E402


def trace_kernels(prof):
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    return [kernel_key(e["name"]) for e in events if e.get("cat") == "kernel"]


class Coverage:
    def __init__(self):
        self.by_kernel = defaultdict(set)

    def add(self, test, keys):
        for k in keys:
            self.by_kernel[k].add(test)

    @pytest.hookimpl(hookwrapper=True)
    def pytest_runtest_call(self, item):
        mod = getattr(item, "module", None)
        helper = getattr(mod, "launched_kernels", None)
        if helper is not None:
            def recording(fn):
                out, ks = helper(fn)
                self.add(item.nodeid, [k for k, _, _ in ks])
                return out, ks

            mod.launched_kernels = recording
            try:
                yield
            finally:
                mod.launched_kernels = helper
            return
        import torch
        from torch.profiler import ProfilerActivity, profile

        if not torch.cuda.is_available():
            yield
            return
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            yield
            torch.cuda.synchronize()
        self.add(item.nodeid, trace_kernels(prof))


def run_in_process(args):
    cov = Coverage()
    rc = pytest.main(["-p", "no:cacheprovider", *args], plugins=[cov])
    return int(rc), {k: sorted(v) for k, v in cov.by_kernel.items()}


def main(argv):
    out_json = None
    if argv[:1] == ["--json"]:
        out_json, argv = argv[1], argv[2:]
    if argv[:1] == ["--one"]:             # child: one pytest run in this process, kernels -> out_json
        rc, seen = run_in_process(argv[1:])
        with open(out_json, "w") as f:
            json.dump(seen, f)
        return rc
    by_kernel, rcs = defaultdict(set), {}
    if argv:
        rc, seen = run_in_process(argv)
        rcs["pytest " + " ".join(argv)] = rc
        for k, v in seen.items():
            by_kernel[k].update(v)
    else:
        tests = os.path.join(ROOT, "tests")
        with tempfile.TemporaryDirectory() as d:
            for name in sorted(f for f in os.listdir(tests) if f.startswith("test_") and f.endswith(".py")):
                part = os.path.join(d, name + ".json")
                rc = subprocess.run([sys.executable, os.path.abspath(__file__), "--json", part, "--one",
                                     os.path.join(tests, name), "-m", "gpu", "-q"], cwd=ROOT).returncode
                rcs[name] = rc
                if os.path.exists(part):
                    with open(part) as f:
                        for k, v in json.load(f).items():
                            by_kernel[k].update(v)
    lib = library_kernels()
    seen = {k: sorted(v) for k, v in by_kernel.items() if k in lib}
    foreign = sorted(k for k in by_kernel if k.startswith("genpc::") and k not in lib)
    failed = {k: v for k, v in rcs.items() if v not in (0, 5)}     # 5: no GPU test in that file
    print(f"\n{len(lib)} instantiations in the library, {len(seen)} launched by the suite; pytest runs that failed: {failed or 'none'}")
    for k in sorted(lib):
        tests = seen.get(k, [])
        print(f"  {'ran ' if tests else '--- '} {k:48s} {KERNELS.get(k, '(no inventory entry)')}"
              + (f"  [{len(tests)} tests, e.g. {tests[0]}]" if tests else ""))
    if foreign:
        print("launched genpc kernels not found in the library (name spelling?):", foreign)
    print("\nnot launched by any test:")
    for k in sorted(lib - set(seen)):
        print(f"  {k:48s} {KERNELS.get(k, '(no inventory entry)')}")
    if out_json:
        with open(out_json, "w") as f:
            json.dump(seen, f, indent=1, sort_keys=True)
    return 1 if failed else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
