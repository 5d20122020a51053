"""The drop-in, pinned against the REAL reference.  tests/golden/reference_dropin.json records every call the reference's own
`torchx.runner.api.Runner` made on this repo's `local_cuda` scheduler while it ran its own `dist.ddp` AppDef (-j 1x2, CPU/gloo
toy job) - once with the factory handed to the Runner (torchx/runner/api.py:621-632) and once with the factory the
reference's registry found in the `torchx_plugins.schedulers` namespace plugin of INTEGRATION.md - with each call's
arguments and results (tests/golden/make_golden.py).  These tests replay those calls, with the reference's AppDef and
resolved cfg rebuilt in this package's types, and require the results the reference saw."""
import json
import os
import re
import time
import textwrap

import pytest

from tests._util import encode
from torchx_b200 import plugins, specs
from torchx_b200.schedulers import api as sched_api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_dropin.json")))

# the INTEGRATION.md plugin, written against this package's plugin namespace and registry
PLUGIN = textwrap.dedent('''
    from torchx_b200.plugins import register


    @register.scheduler(name="local_cuda")
    def local_cuda(session_name: str, **kwargs):
        from torchx_b200.schedulers.local_cuda_scheduler import create_scheduler
        return create_scheduler(session_name, **kwargs)


    @register.scheduler(name="local_cwd")
    def local_cwd(session_name: str, **kwargs):
        from torchx_b200.schedulers.local_scheduler import create_scheduler
        return create_scheduler(session_name, **kwargs)
''')


def _decode(v, tokens, dryrun):
    if isinstance(v, dict):
        if "__enum__" in v:
            cls, name = v["__enum__"]
            return getattr(getattr(specs, cls, None) or getattr(sched_api, cls), name)
        if "__dataclass__" in v:
            cls = getattr(specs, v["__dataclass__"], None) or getattr(sched_api, v["__dataclass__"])
            return cls(**{k: _decode(x, tokens, dryrun) for k, x in v["fields"].items()})
        if "__object__" in v:
            assert v["__object__"] == "AppDryRunInfo", v
            return dryrun
        return {k: _decode(x, tokens, dryrun) for k, x in v.items()}
    if isinstance(v, list):
        return [_decode(x, tokens, dryrun) for x in v]
    if isinstance(v, str):
        for tok, real in tokens.items():
            v = v.replace(tok, real)
    return v


def _mask_digest(lines):
    return [re.sub(r"sha256 [0-9a-f]{16}", "sha256 <digest>", ln) for ln in lines]  # host-CPU float math, not the scheduler


def _replay(trace, factory, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("PYTHONPATH", ROOT)  # the toy job imports torchx_b200.distributed
    tokens = {"<script>": os.path.join(ROOT, "examples", "toy_ddp.py"), "<log_dir>": str(tmp_path / "logs"),
              "<home>": str(tmp_path / "home")}
    monkeypatch.setenv("TORCHX_HOME", tokens["<home>"])  # as when the trace was recorded: the app registry lives there
    fc = trace["factory_call"]
    sched = factory(fc["session_name"], **_decode(fc["kwargs"], tokens, None))
    dryrun = None
    try:
        for call in trace["calls"]:
            method, want = call["method"], call["result"]
            args = _decode(call["args"], tokens, dryrun)
            kwargs = _decode(call["kwargs"], tokens, dryrun)
            res = getattr(sched, method)(*args, **kwargs)
            if method == "schedule":
                assert res.startswith(trace["describe_roles"][0] + "-"), res
                tokens["<app_id>"] = res
            subst = {real: tok for tok, real in tokens.items()}
            got = encode(list(res) if method == "log_iter" else res, subst)
            if method == "submit_dryrun":
                dryrun = res
            elif method == "describe":  # the Runner's status polls: wait for terminal states, accept any while running
                state = specs.AppState[want["fields"]["state"]["__enum__"][1]]
                deadline = time.monotonic() + 300
                while state in (specs.AppState.SUCCEEDED, specs.AppState.FAILED) and res.state != state:
                    assert res.state not in (specs.AppState.SUCCEEDED, specs.AppState.FAILED, specs.AppState.CANCELLED), got
                    assert time.monotonic() < deadline, got
                    time.sleep(0.2)
                    res = sched.describe(*args)
                    got = encode(res, subst)
                got["fields"].pop("state")
                want = {**want, "fields": {k: x for k, x in want["fields"].items() if k != "state"}}
            elif method == "log_iter":
                got, want = _mask_digest(got), _mask_digest(want)
            assert got == want, (method, got, want)
    finally:
        sched.close()
    assert trace["state"] == "SUCCEEDED" and trace["handle"] == "local_cuda://torchx/<app_id>"


def test_reference_runner_drives_local_cuda_through_the_factory(tmp_path, monkeypatch):
    from torchx_b200.schedulers.local_cuda_scheduler import create_scheduler

    _replay(G["factory"], create_scheduler, tmp_path, monkeypatch)


def test_reference_registry_finds_local_cuda_as_a_namespace_plugin(tmp_path, monkeypatch):
    pkg = tmp_path / "plug" / "torchx_b200_plugins" / "schedulers"
    pkg.mkdir(parents=True)
    (pkg / "b200.py").write_text(PLUGIN)  # namespace packages: no __init__.py on purpose
    monkeypatch.syspath_prepend(str(tmp_path / "plug"))
    plugins.reset_for_tests()
    try:
        from torchx_b200.schedulers import get_scheduler_factories

        # the defaults carry the same two names: require that the registry found them in the plugin module
        assert sorted(plugins.registered_schedulers()) == G["plugin"]["schedulers"]
        factories = get_scheduler_factories()
        assert sorted(factories) == G["plugin"]["schedulers"]
        assert {f.__module__ for f in factories.values()} == {"torchx_b200_plugins.schedulers.b200"}
        _replay(G["plugin"], factories["local_cuda"], tmp_path, monkeypatch)
    finally:
        monkeypatch.undo()
        plugins.reset_for_tests()
