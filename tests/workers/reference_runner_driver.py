"""Runs INSIDE a subprocess whose sys.path has the reference TorchX checkout first: the REFERENCE's own Runner / scheduler
registry drives this repo's `local_cuda` scheduler through a tracing proxy, and every call the Runner makes on the
scheduler (arguments and results) is written as JSON to ``out_path``.  tests/golden/make_golden.py stores the trace as
tests/golden/reference_dropin.json; tests/test_reference_dropin.py replays it without the reference.

    python reference_runner_driver.py {factory|plugin} <script> <log_dir> <out_path>
"""
import json
import os
import sys

mode, script, log_dir, out_path = sys.argv[1:5]

import torchx  # noqa: E402  (the reference package)
from torchx.runner.api import Runner  # noqa: E402
from torchx.specs import AppState  # noqa: E402

from tests._util import encode  # noqa: E402

ref_root = os.path.dirname(os.path.dirname(os.path.realpath(torchx.__file__)))
dist_ddp = os.path.join(ref_root, "torchx", "components", "dist.py") + ":ddp"  # builtin-by-name discovery needs hydra (SURVEY 8c)
subst = {script: "<script>", log_dir: "<log_dir>", os.environ["TORCHX_HOME"]: "<home>"}


def enc(v):
    return encode(v, subst)


class Tracer:
    """Forwards every attribute to the scheduler and records the public method calls made through it."""

    def __init__(self, inner, calls):
        self._inner, self._calls = inner, calls

    def __getattr__(self, name):
        attr = getattr(self._inner, name)
        if not callable(attr):
            return attr

        def call(*args, **kwargs):
            rec = {"method": name, "args": enc(args), "kwargs": enc(kwargs)}
            self._calls.append(rec)
            res = attr(*args, **kwargs)
            if name == "schedule":
                subst[res] = "<app_id>"
            if name == "log_iter":
                lines = list(res)
                rec["result"] = enc(lines)
                return iter(lines)
            rec["result"] = enc(res)
            return res

        return call


calls = []
out = {"mode": mode}

if mode == "factory":
    # torchx/runner/api.py:621-632: a Runner is handed {name: factory}; ours has the reference factory signature
    from torchx_b200.schedulers.local_cuda_scheduler import create_scheduler

    def traced_factory(session_name, **kwargs):
        out["factory_call"] = {"session_name": session_name, "kwargs": enc(kwargs)}
        return Tracer(create_scheduler(session_name, **kwargs), calls)

    runner = Runner("torchx", {"local_cuda": traced_factory})
elif mode == "plugin":
    # torchx/schedulers/__init__.py:40-60: the registry the CLI uses; the torchx_plugins namespace package on sys.path
    # (written by make_golden.py from INTEGRATION.md) registers local_cuda (and re-registers local_cwd)
    from torchx.schedulers import get_scheduler_factories

    factories = get_scheduler_factories()
    out["schedulers"] = sorted(factories)
    assert "local_cuda" in factories and "local_cwd" in factories, sorted(factories)
    found = factories["local_cuda"]

    def traced_factory(session_name, **kwargs):
        out["factory_call"] = {"session_name": session_name, "kwargs": enc(kwargs)}
        return Tracer(found(session_name, **kwargs), calls)

    runner = Runner("torchx", {**factories, "local_cuda": traced_factory})
else:
    raise SystemExit(mode)

with runner:
    cfg = {"log_dir": log_dir}
    dry = runner.dryrun_component(dist_ddp, ["-j", "1x2", "--script", script], "local_cuda", cfg)
    out["dryrun_repr_has_workers"] = "RANK" in repr(dry) or "rank" in repr(dry).lower()
    handle = runner.run_component(dist_ddp, ["-j", "1x2", "--script", script], "local_cuda", cfg)
    status = runner.wait(handle, wait_interval=0.2)
    out["state"] = status.state.name
    out["ok"] = status.state == AppState.SUCCEEDED
    out["describe_roles"] = [r.name for r in runner.describe(handle).roles] if runner.describe(handle) else None
    out["log_tail"] = [ln.rstrip("\n") for ln in runner.log_lines(handle, "toy_ddp", 0)][-4:]
    out["list"] = [enc(a.app_id) for a in runner.list("local_cuda")][:3]
    out["handle"] = enc(handle)
out["calls"] = []
for c in calls:  # the Runner's status polls: one entry per run of identical calls
    if out["calls"] and {k: v for k, v in out["calls"][-1].items() if k != "times"} == c:
        out["calls"][-1]["times"] += 1
    else:
        out["calls"].append({**c, "times": 1})
with open(out_path, "w") as f:
    json.dump(out, f, indent=1, sort_keys=True)
print(json.dumps({"ok": out["ok"], "calls": len(calls)}))
