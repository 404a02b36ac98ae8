"""Which kernel instantiations of libmridc_b200.so the GPU suite launches.

Runs `pytest -m gpu` in this process with a plugin that records every test's CUDA kernels with torch.profiler (CUPTI), then
compares the names with the library's inventory (tests/test_gpu_kernel_paths.py: cuobjdump -elf + GNU c++filt).  Prints the
count for the whole suite, the count without tests/test_gpu_kernel_paths.py (the suite before that file existed) and the
instantiations nothing launched.  The rows of test_gpu_kernel_paths.py run their own profiler sessions (sessions do not
nest): for them the plugin collects what those sessions record, through the module's KERNEL_SINK.

    python tools/kernel_coverage.py [--json FILE] [extra pytest arguments]   # run (part of) the suite, optionally save
    python tools/kernel_coverage.py --merge FILE [FILE ...]                  # counts over saved runs
"""
import json
import os
import sys

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

PATHS_FILE = "test_gpu_kernel_paths.py"


class KernelRecorder:
    def __init__(self, kernel_name):
        self.kernel_name = kernel_name
        self.by_test = {}

    @pytest.hookimpl(hookwrapper=True)
    def pytest_runtest_call(self, item):
        from torch.profiler import ProfilerActivity, profile

        mod = getattr(item, "module", None)
        if mod is not None and hasattr(mod, "KERNEL_SINK"):
            mod.KERNEL_SINK = sink = set()
            try:
                yield
            finally:
                mod.KERNEL_SINK = None
            self.by_test[item.nodeid] = set(sink)
            return
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            yield
            if torch.cuda.is_initialized():
                torch.cuda.synchronize()
        names = {self.kernel_name(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        self.by_test[item.nodeid] = {n for n in names if n.startswith("mrb::")}


def report(by_test, inv):
    every = set().union(*by_test.values()) if by_test else set()
    before = set().union(*[v for k, v in by_test.items() if PATHS_FILE not in k]) if by_test else set()
    print("\nkernel instantiations in libmridc_b200.so: %d" % len(inv))
    print("launched by the GPU suite without %s: %d / %d" % (PATHS_FILE, len(before & inv), len(inv)))
    print("launched by the whole GPU suite: %d / %d" % (len(every & inv), len(inv)))
    for n in sorted(inv - every):
        print("  never launched: %s" % n)


def main(argv):
    from test_gpu_kernel_paths import kernel_name, library_instantiations

    inv = set(library_instantiations())
    if argv[:1] == ["--merge"]:
        by_test = {}
        for path in argv[1:]:
            with open(path) as fh:
                by_test.update({k: set(v) for k, v in json.load(fh).items()})
        report(by_test, inv)
        return 0
    out = None
    if argv[:1] == ["--json"]:
        out, argv = argv[1], argv[2:]
    rec = KernelRecorder(kernel_name)
    rc = pytest.main(["-q", "-m", "gpu", "-p", "no:cacheprovider", os.path.join(REPO, "tests")] + argv, plugins=[rec])
    if out:
        with open(out, "w") as fh:
            json.dump({k: sorted(v) for k, v in rec.by_test.items()}, fh, indent=1)
    report(rec.by_test, inv)
    return int(rc)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
