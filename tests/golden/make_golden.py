"""Generates the committed golden fixtures by RUNNING THE REFERENCE in the build container.

  ddp_w{2,4}.npz   stock torch DistributedDataParallel (no hook / allreduce_hook / bf16_compress_hook) launched
                   through the reference's own launcher:  PYTHONPATH=/root/reference python -m torchx.cli.main
                   run -s local_cwd /root/reference/torchx/components/dist.py:ddp -j 1xW --script <worker>
                   (gloo/CPU - there is no GPU here; SURVEY.md §8c, Appendix C).  Holds every rank's local
                   gradients and the three averaged results, so the oracle can be pinned against them.
  bucket_layouts.json   torch's own dist._compute_bucket_assignment_by_size over ResNet-50 / GPT-2-small /
                   BERT-base parameters (reverse order, limits [1 MiB, 25 MiB]) - layout parity fixture.
  reference_dropin.json   every call the reference's own Runner makes on the local_cuda scheduler (factory handed to
                   the Runner, and found as a torchx_plugins namespace plugin), with arguments and results.

Run from the repo root:  python tests/golden/make_golden.py      (needs /root/reference; not needed at test time)
"""
import json
import os
import subprocess
import sys
import tempfile
import textwrap

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"

WORKER = textwrap.dedent(
    '''
    import os, sys, argparse
    import numpy as np
    import torch, torch.nn as nn, torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    from torch.distributed.algorithms.ddp_comm_hooks import default_hooks

    ap = argparse.ArgumentParser(); ap.add_argument("--out"); a = ap.parse_args()
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()

    def model():
        torch.manual_seed(0)
        return nn.Sequential(nn.Linear(64, 128), nn.ReLU(), nn.Linear(128, 16))

    torch.manual_seed(100 + rank)
    x = torch.randn(32, 64)

    def flat_grads(m):
        return torch.cat([p.grad.reshape(-1) for p in m.parameters()])

    m = model(); m(x).sum().backward(); local = flat_grads(m).clone()
    gathered = [torch.empty_like(local) for _ in range(world)]
    dist.all_gather(gathered, local)

    res = {}
    for name, hook in (("none", None), ("allreduce", default_hooks.allreduce_hook), ("bf16_compress", default_hooks.bf16_compress_hook)):
        d = DDP(model())
        if hook is not None:
            d.register_comm_hook(None, hook)
        d(x).sum().backward()
        res[name] = flat_grads(d.module).clone()
        dist.barrier()
    outs = {}
    for k, v in res.items():
        g = [torch.empty_like(v) for _ in range(world)]
        dist.all_gather(g, v)
        outs[k] = torch.stack(g).numpy()
    if rank == 0:
        np.savez(a.out, local=torch.stack(gathered).numpy(), **{"ddp_" + k: v for k, v in outs.items()})
    dist.barrier()
    dist.destroy_process_group()
    '''
)


def run_reference_ddp(world: int) -> None:
    out = os.path.join(HERE, f"ddp_w{world}.npz")
    with tempfile.TemporaryDirectory() as td:
        script = os.path.join(td, "golden_worker.py")
        with open(script, "w") as f:
            f.write(WORKER)
        env = dict(os.environ, PYTHONPATH=REF)
        cmd = [sys.executable, "-m", "torchx.cli.main", "run", "-s", "local_cwd", f"{REF}/torchx/components/dist.py:ddp",
               "-j", f"1x{world}", "--script", script, "--", "--out", out]
        subprocess.run(cmd, check=True, cwd=td, env=env)
    assert os.path.exists(out), out
    print("wrote", out)


def bucket_layouts() -> None:
    import torch
    import torch.distributed as dist

    def layout(params):
        rev = list(reversed(range(len(params))))
        idx, _ = dist._compute_bucket_assignment_by_size([params[i] for i in rev], [1024 * 1024, 25 * 1024 * 1024], [False] * len(rev), rev)
        return idx

    out = {}
    import torchvision

    models = {"resnet50": lambda: torchvision.models.resnet50()}
    try:
        from transformers import BertConfig, BertForMaskedLM, GPT2Config, GPT2LMHeadModel

        models["gpt2_small"] = lambda: GPT2LMHeadModel(GPT2Config())
        models["bert_base"] = lambda: BertForMaskedLM(BertConfig())
    except Exception as e:  # pragma: no cover
        print("transformers unavailable:", e)
    for name, ctor in models.items():
        with torch.device("meta"):
            m = ctor()
        params = [p for p in m.parameters() if p.requires_grad]
        real = [torch.empty(p.shape, dtype=torch.float32, device="meta") for p in params]
        out[name] = {
            "param_numel": [p.numel() for p in params],
            "buckets_fp32": layout(real),
            "buckets_bf16": layout([torch.empty(p.shape, dtype=torch.bfloat16, device="meta") for p in params]),
        }
        print(name, "params", len(params), "numel", sum(out[name]["param_numel"]), "buckets", len(out[name]["buckets_fp32"]))
    with open(os.path.join(HERE, "bucket_layouts.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))


def launcher_goldens() -> None:
    """What the REFERENCE launcher produces for the inputs our launcher tests use: dist.ddp AppDefs, -j parsing,
    cfg-string parsing, macro substitution, local_cwd dry-run requests, CUDA_VISIBLE_DEVICES tables."""
    sys.path.insert(0, REF)
    from dataclasses import asdict
    from unittest import mock

    from torchx.components.dist import ddp, parse_nnodes
    from torchx.components.structured_arg import StructuredNameArgument
    from torchx.schedulers.local_scheduler import create_scheduler, Opts
    from torchx.specs import AppDef, Resource, Role, macros, runopts
    from torchx.util.types import to_dict

    out = {}
    cases = {
        "script_1x8": dict(args=["--foo", "bar"], kw=dict(script="toy_ddp.py", j="1x8", gpu=8)),
        "module_elastic": dict(args=[], kw=dict(m="pkg.train.main", j="1:2x4", h="gpu.large", name="exp/run1", max_retries=3,
                                                 env={"A": "1"}, rdzv_conf="join_timeout=600")),
        "single_proc_debug": dict(args=["--x=1"], kw=dict(script="a/b/train.py", j="2", debug=True, name="myexp/", tee=1)),
        "static_rdzv": dict(args=[], kw=dict(script="t.py", j="2x2", rdzv_backend="static", rdzv_port=12345)),
    }
    with mock.patch.dict(os.environ, {"LOGLEVEL": "WARNING"}):
        for name, c in cases.items():
            app = ddp(*c["args"], **c["kw"])
            d = asdict(app)
            for r in d["roles"]:
                r.pop("overrides", None)
                r.pop("workspace", None)
                r.pop("mounts", None)
                r["resource"] = {k: r["resource"][k] for k in ("cpu", "gpu", "memMB")}
                r["retry_policy"] = str(r["retry_policy"].value)
                r.pop("image", None)
            out.setdefault("ddp", {})[name] = {"call": {"args": c["args"], "kw": c["kw"]}, "app": d}
    out["parse_nnodes"] = {j: list(parse_nnodes(j)) for j in ("2", "1x2", "1:2x3", "4x8", "0:1x2")}
    out["name_arg"] = {
        f"{n}|{m}|{s}": asdict(StructuredNameArgument.parse_from(name=n, m=m, script=s))
        for n, m, s in (("foo/bar", None, "bar/baz.py"), ("foo/", None, "bar/baz.py"), ("/bar", None, "bar/baz.py"),
                        ("foobar", "foo.bar", None), ("foo/", "foo.bar.baz", None), ("/", None, "x/y/z.py"))
    }
    out["to_dict"] = {lit: to_dict(lit) for lit in ("", "FOO=v1", "FOO=''", "FOO=v1,v2", "FOO=v1;v2", "FOO=v1,v2,BAR=v3",
                                                    "FOO=v1;v2,BAR=v3", "FOO=v1;v2;BAR=v3", 'FOO="value with = and , and ;"',
                                                    "log_dir=/tmp/x,prepend_cwd=True")}
    opts = runopts()
    from typing import Dict, List

    opts.add("FOO", type_=List[str], default=["a"], help="list")
    opts.add("BAR", type_=str, required=True, help="str")
    opts.add("N", type_=int, default=3, help="int")
    opts.add("B", type_=bool, default=False, help="bool")
    opts.add("D", type_=Dict[str, str], default=None, help="dict")
    out["cfg_from_str"] = {lit: opts.cfg_from_str(lit) for lit in ("", "FOO=v1", "FOO=v1,v2", "FOO=v1;v2,BAR=v3", "N=7,B=true,BAR=x",
                                                                    "D=a:1;b:2,BAR=y")}
    out["resolve"] = opts.resolve({"BAR": "z"})
    role = Role(name="r", image="img", entrypoint="e", args=["${img_root}/x", "--id", "${app_id}", "${replica_id}", "$$lit", "${unknown}"],
                env={"H": "${rank0_env}"}, metadata={"k": {"a": ["${app_id}", {"b": "${replica_id}"}]}}, resource=Resource(1, 0, 1))
    rr = macros.Values(img_root="/img", app_id="app-1", replica_id="3", rank0_env="TORCHX_RANK0_HOST").apply(role)
    out["macros"] = {"args": rr.args, "env": rr.env, "metadata": rr.metadata}

    # CUDA_VISIBLE_DEVICES partitioning table (reference local_scheduler_test.py:915-1113 scenarios)
    def cvd(device_count, roles, auto=True):
        sched = create_scheduler("golden")
        try:
            with mock.patch.object(sched, "_cuda_device_count", return_value=device_count):
                app = AppDef("a", roles=[Role(name=n, image="", entrypoint="e", num_replicas=k, resource=Resource(1, g, 1)) for n, k, g in roles])
                info = sched.submit_dryrun(app, {"auto_set_cuda_visible_devices": auto})
                return {n: [p.env.get("CUDA_VISIBLE_DEVICES") for p in info.request.role_params[n]] for n, _, _ in roles}
        finally:
            sched.close()

    out["cuda_visible_devices"] = {
        "8gpu_1role_2x4": cvd(8, [("t", 2, 4)]),
        "8gpu_2roles": cvd(8, [("a", 1, 2), ("b", 3, 2)]),
        "8gpu_too_many": cvd(8, [("t", 3, 4)]),
        "0gpu": cvd(0, [("t", 1, 2)]),
        "16gpu_cpu_and_gpu_roles": cvd(16, [("cpu", 2, 0), ("g", 2, 8)]),
        "8gpu_auto_off": cvd(8, [("t", 2, 4)], auto=False),
    }

    # a local_cwd dry-run request for the unmodified dist.ddp AppDef (env additions + log file layout)
    sched = create_scheduler("golden")
    try:
        app = ddp("--foo", "bar", script="toy_ddp.py", j="1x2")
        info = sched.submit_dryrun(app, {"log_dir": "/tmp/golden_logs"})
        req = info.request
        rp = req.role_params["toy_ddp"][0]
        out["local_cwd_request"] = {
            "args": [a.replace(req.app_id, "<APP_ID>") for a in rp.args],
            "env_added": {k: v.replace(req.app_id, "<APP_ID>") for k, v in rp.env.items() if k in ("TORCHX_RANK0_HOST", "TORCHELASTIC_ERROR_FILE", "PET_LOG_DIR")},
            "stdout": rp.stdout.replace(req.app_id, "<APP_ID>"), "stderr": rp.stderr.replace(req.app_id, "<APP_ID>"),
            "combined": rp.combined.replace(req.app_id, "<APP_ID>"), "log_dir": req.log_dir.replace(req.app_id, "<APP_ID>"),
            "created_dirs": os.path.exists(req.log_dir),
        }
    finally:
        sched.close()
    with open(os.path.join(HERE, "launcher.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote launcher.json")


DROPIN_PLUGIN = textwrap.dedent('''
    from torchx.plugins import register


    @register.scheduler(name="local_cuda")
    def local_cuda(session_name: str, **kwargs):
        from torchx_b200.schedulers.local_cuda_scheduler import create_scheduler
        return create_scheduler(session_name, **kwargs)


    @register.scheduler(name="local_cwd")
    def local_cwd(session_name: str, **kwargs):
        from torchx.schedulers.local_scheduler import create_scheduler
        return create_scheduler(session_name, **kwargs)
''')


def dropin_traces() -> None:
    """The reference's own Runner submits its own dist.ddp AppDef (-j 1x2, CPU/gloo toy job) to local_cuda, once with the
    factory handed to the Runner and once through the torchx_plugins namespace plugin of INTEGRATION.md; every call the
    Runner makes on the scheduler is recorded (tests/workers/reference_runner_driver.py)."""
    root = os.path.dirname(os.path.dirname(HERE))
    out = {}
    for mode in ("factory", "plugin"):
        with tempfile.TemporaryDirectory() as td:
            extra = []
            if mode == "plugin":
                pkg = os.path.join(td, "plug", "torchx_plugins", "schedulers")
                os.makedirs(pkg)
                with open(os.path.join(pkg, "b200.py"), "w") as f:  # namespace packages: no __init__.py on purpose
                    f.write(DROPIN_PLUGIN)
                extra = [os.path.join(td, "plug")]
            env = dict(os.environ, PYTHONPATH=os.pathsep.join([REF, *extra, root]), TORCHX_HOME=os.path.join(td, "home"))
            trace = os.path.join(td, "trace.json")
            cmd = [sys.executable, os.path.join(root, "tests", "workers", "reference_runner_driver.py"), mode,
                   os.path.join(root, "examples", "toy_ddp.py"), os.path.join(td, "logs"), trace]
            subprocess.run(cmd, check=True, cwd=td, env=env, timeout=600)
            with open(trace) as f:
                out[mode] = json.load(f)
    with open(os.path.join(HERE, "reference_dropin.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote reference_dropin.json")


if __name__ == "__main__":
    what = sys.argv[1:] or ["ddp", "buckets", "launcher", "dropin"]
    if "ddp" in what:
        for w in (2, 4):
            run_reference_ddp(w)
    if "buckets" in what:
        bucket_layouts()
    if "launcher" in what:
        launcher_goldens()
    if "dropin" in what:
        dropin_traces()
