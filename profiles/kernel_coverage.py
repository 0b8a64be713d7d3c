"""Which CUDA kernels a pytest selection launches, and how often.

Runs pytest in this process inside one torch.profiler session (CUDA activities) and writes the
sorted kernel names with their launch counts as JSON. With --baseline (the JSON of an earlier run,
e.g. the suite without a new test file) the output also lists the kernels this run launched and the
baseline did not: the instantiations only the added tests reach.

    python profiles/kernel_coverage.py --out DIR --name NAME [--baseline FILE] -- -m gpu tests/...

Kernels of bench.py's subprocess are not seen (another process). Tests that run their own
profiler session (tests/test_gpu_sdf_thresholds.py) see VGT_B200_KERNEL_COVERAGE=1 and leave
the profiler to this script.
"""
import argparse
import json
import os
import sys
from pathlib import Path

REPO = Path(__file__).resolve().parents[1]


def short_name(name: str) -> str:
    name = name.replace("(anonymous namespace)::", "")
    if name.startswith("void "):
        name = name[len("void "):]
    return name.split("(")[0]


def main() -> int:
    parser = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    parser.add_argument("--out", required=True, help="output directory")
    parser.add_argument("--name", default="kernel_coverage")
    parser.add_argument("--baseline", help="JSON written by an earlier run of this script")
    parser.add_argument("pytest_args", nargs=argparse.REMAINDER)
    args = parser.parse_args()
    pytest_args = [a for a in args.pytest_args if a != "--"]

    import pytest
    import torch
    os.environ["VGT_B200_KERNEL_COVERAGE"] = "1"
    os.chdir(REPO)
    torch.cuda.init()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as profile:
        exit_code = int(pytest.main(pytest_args))
        torch.cuda.synchronize()
    kernels = {}
    for event in profile.events():
        if event.device_type == torch.autograd.DeviceType.CUDA and not event.name.startswith(
                ("Memcpy", "Memset")):
            name = short_name(event.name)
            kernels[name] = kernels.get(name, 0) + 1
    result = {
        "pytest_args": pytest_args,
        "pytest_exit_code": exit_code,
        "device": torch.cuda.get_device_name(0),
        "kernels": dict(sorted(kernels.items())),
    }
    if args.baseline:
        baseline = json.loads(Path(args.baseline).read_text())
        result["baseline_pytest_args"] = baseline["pytest_args"]
        result["not_in_baseline"] = sorted(set(kernels) - set(baseline["kernels"]))
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / f"{args.name}.json").write_text(json.dumps(result, indent=1) + "\n")
    print(f"{len(kernels)} kernels, {sum(kernels.values())} launches -> {out / args.name}.json")
    return exit_code


if __name__ == "__main__":
    sys.exit(main())
