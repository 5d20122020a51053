#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): images/sec of ResNet-50 DDP training on N B200s of one box.

    python bench.py --gpus 1 --steps K --warmup W                      # N=1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                         # N>1, one rank per GPU
    ... --impl reference                                                # the reference path, same workload

A step = one optimizer step on a synthetic ImageNet-shaped batch (B=256/GPU, bf16 autocast, channels_last, SGD
momentum) of random-init torchvision ResNet-50 (BASELINE.md config #2): forward, backward with the DDP gradient-
bucket averaging (5 buckets, 97.5 MiB fp32) overlapped, optimizer step.

  default arm   torchx_b200.ddp.DistributedDataParallel: every bucket averaged by ONE fused sm_100a kernel
                (libb200ddp.so) over NVSwitch peer buffers / NVLS multicast; no torch.distributed / NCCL anywhere.
  reference arm what `torchx run -s local_cwd dist.ddp` workers run: stock torch DistributedDataParallel over NCCL
                with bf16_compress_hook (cast, div, ncclAllReduce, copy per bucket).
  --impl reference_tuned   the same with gradient_as_bucket_view=True, static_graph=True (attribution arm, not the headline)
  --model gpt2 | bert      BASELINE.json configs[2] / configs[4]: GPT2LMHeadModel(GPT2Config()) on [8,1024] tokens,
                BertForMaskedLM(BertConfig()) on [16,512] tokens, AdamW; the metric becomes sequences/sec.

`value` is measured with the batch resident in HBM; `e2e` through the public API with the batch coming from pinned
host memory every step (H2D inside the timed region, overlapped on a copy stream) and the loss read back (D2H).
Both are device-timed with CUDA events, barrier + synchronize on both sides, max over ranks.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference_tuned"])
    ap.add_argument("--batch", type=int, default=0, help="samples per GPU per step (default: 256 images / 8 GPT-2 sequences / 16 BERT sequences)")
    ap.add_argument("--model", default="resnet50", choices=["resnet50", "gpt2", "bert"])
    ap.add_argument("--no-parity", dest="parity", action="store_false", help="(N>1) skip the oracle parity check of the bucket allreduce")
    ap.add_argument("--wire", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sweep", action="store_true", default=True, help="(N>1) also report allreduce bus GB/s at the model's bucket sizes and 256 MiB")
    ap.add_argument("--no-sweep", dest="sweep", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed on rank 0 as DIR/<name>.npy (float32): loss, logits, "
                         "the averaged gradients and the updated parameters; arrays over %d elements as the same seeded sample "
                         "of positions in every run, so two builds can be compared output for output.  Such a run uses deterministic "
                         "cuDNN / cuBLAS algorithms instead of autotuned ones, so its timing is not the headline number; two such runs "
                         "of one build on the same GPU model and library versions give the same bits, other GPUs or libraries need not" % (1 << 21))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1: the timed region is --steps optimizer steps")
    return args


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int) -> None:
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
                pw.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "power_w_max": max(pw) if pw else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


MODELS = {
    "resnet50": {"batch": 256, "unit": "images", "metric": "images/sec (max over ranks) ResNet-50 DDP", "opt": "sgd",
                 "workload": "ResNet-50 bf16 dist.ddp training step (BASELINE.json configs[1]), B=%d/GPU, 3x224x224, channels_last, SGD momentum"},
    "gpt2": {"batch": 8, "unit": "sequences", "metric": "sequences/sec (max over ranks) GPT-2-small DDP", "opt": "adamw", "seq": 1024, "vocab": 50257,
             "workload": "GPT-2-small (GPT2LMHeadModel(GPT2Config())) bf16 dist.ddp training step (BASELINE.json configs[2]), B=%d x 1024 tokens/GPU, AdamW"},
    "bert": {"batch": 16, "unit": "sequences", "metric": "sequences/sec (max over ranks) BERT-base DDP", "opt": "adamw", "seq": 512, "vocab": 30522,
             "workload": "BERT-base (BertForMaskedLM(BertConfig())) bf16 dist.ddp training step (BASELINE.json configs[4]), B=%d x 512 tokens/GPU, AdamW"},
}


def build_model(name: str, device):
    import torch

    torch.manual_seed(0)  # identical init on every rank (then rank-0 broadcast, as DDP does)
    if name == "resnet50":
        import torchvision

        return torchvision.models.resnet50().to(device).to(memory_format=torch.channels_last)
    import transformers

    transformers.logging.set_verbosity_error()
    if name == "gpt2":
        m = transformers.GPT2LMHeadModel(transformers.GPT2Config())
    elif name == "bert":
        m = transformers.BertForMaskedLM(transformers.BertConfig())
    else:
        raise SystemExit(f"unknown model {name}")
    return m.to(device)


def synthetic_batches(model: str, batch: int, rank: int, count: int, pinned: bool):
    """(input, target) pairs on the host: ImageNet-shaped images + labels, or token ids + LM / MLM labels."""
    import torch

    g = torch.Generator().manual_seed(1000 + rank)
    out = []
    for _ in range(count):
        if model == "resnet50":
            x = torch.randn(batch, 3, 224, 224, generator=g)
            y = torch.randint(0, 1000, (batch,), generator=g)
        else:
            spec = MODELS[model]
            x = torch.randint(0, spec["vocab"], (batch, spec["seq"]), generator=g)
            y = x.clone() if model == "gpt2" else torch.randint(0, spec["vocab"], (batch, spec["seq"]), generator=g)
        if pinned:
            x, y = x.pin_memory(), y.pin_memory()
        out.append((x, y))
    return out


def planned_bucket_sizes_mib(model):
    """The gradient-bucket layout both arms end up with (reverse parameter order, 1 MiB first bucket, 25 MiB cap:
    torchx_b200/ddp/bucketing.py is index-for-index torch's _compute_bucket_assignment_by_size, tests/test_ddp_layout.py)."""
    from torchx_b200.ddp.bucketing import MIB, plan_buckets

    ps = [p for p in model.parameters() if p.requires_grad]
    specs = plan_buckets([p.numel() for p in ps], [p.element_size() for p in ps], [str(p.dtype) for p in ps])
    return [round(sp.nbytes / MIB, 2) for sp in specs]


def nvlink_bytes(gpu: int):
    """(tx, rx) bytes summed over the GPU's NVLinks from `nvidia-smi nvlink -gt d` (hardware counters), or None."""
    import re

    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(gpu)], capture_output=True, text=True, timeout=20).stdout
    except Exception:  # noqa: BLE001
        return None
    tx = sum(int(m) for m in re.findall(r"Data Tx:\s*(\d+)\s*KiB", out))
    rx = sum(int(m) for m in re.findall(r"Data Rx:\s*(\d+)\s*KiB", out))
    return (tx * 1024, rx * 1024) if (tx or rx) else None


class Trainer:
    """The user-level training loop, identical for both arms apart from how the model is wrapped."""

    def __init__(self, args, rank, world, local_rank):
        import torch

        self.torch = torch
        self.args, self.rank, self.world = args, rank, world
        self.device = torch.device("cuda", local_rank)
        torch.cuda.set_device(self.device)
        torch.backends.cudnn.benchmark = not args.dump_outputs
        if args.dump_outputs:
            # the autotuner picks algorithms by timing, and SGD at lr 0.1 grows the last-bit differences between two picks into
            # different weights within the timed steps (ResNet-50, --steps 20 --warmup 5 on a B200 at 1000 W: two autotuned runs
            # ended at loss 5.56 and 3.72): fixed deterministic algorithms make two runs, and two builds, comparable.  Not
            # warn_only: with it cuDNN attention's backward stays non-deterministic (GPT-2 dumps differed), and an op that has
            # no deterministic implementation must stop the run rather than break the promise silently
            torch.backends.cudnn.deterministic = True
            torch.use_deterministic_algorithms(True)
        self.comm = None
        self.is_image = args.model == "resnet50"
        model = build_model(args.model, self.device)
        self.bucket_sizes = planned_bucket_sizes_mib(model)
        if args.impl == "b200":
            from torchx_b200.ddp import Communicator, DistributedDataParallel

            self.comm = Communicator.from_env()
            self.ddp = DistributedDataParallel(model, self.comm, wire=args.wire)
        else:
            import torch.distributed as dist
            from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
            from torch.nn.parallel import DistributedDataParallel as TorchDDP

            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            if "MASTER_PORT" not in os.environ:  # plain `python bench.py --impl reference` (N=1): any free port
                import socket

                with socket.socket() as sock:
                    sock.bind(("127.0.0.1", 0))
                    os.environ["MASTER_PORT"] = str(sock.getsockname()[1])
            # keep stdout to the ONE JSON line: this image's NCCL otherwise prints "NCCL version ..." there
            if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
                os.environ["NCCL_DEBUG"] = "WARN"
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=self.device)
            tuned = {"gradient_as_bucket_view": True, "static_graph": True} if args.impl == "reference_tuned" else {}
            self.ddp = TorchDDP(model, device_ids=[local_rank], **tuned)
            if args.wire == "bf16":
                self.ddp.register_comm_hook(None, default_hooks.bf16_compress_hook)
        if MODELS[args.model]["opt"] == "sgd":
            self.opt = torch.optim.SGD(self.ddp.parameters(), lr=0.1, momentum=0.9)
        else:
            self.opt = torch.optim.AdamW(self.ddp.parameters(), lr=1e-4)
        self.loss_fn = torch.nn.CrossEntropyLoss()
        self.copy_stream = torch.cuda.Stream(device=self.device)

    # -- collective helpers that work for both arms ---------------------------------------------------------
    def barrier(self):
        torch = self.torch
        if self.comm is not None:
            self.comm.barrier()
        elif self.world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, value: float) -> float:
        torch = self.torch
        if self.world == 1:
            return value
        t = torch.zeros(self.world, device=self.device)
        t[self.rank] = value
        if self.comm is not None:
            self.comm.allreduce_(t, scale=1.0, wire="f32")
        else:
            import torch.distributed as dist

            dist.all_reduce(t)
        torch.cuda.synchronize()
        return float(t.max().item())

    # -- one optimizer step -----------------------------------------------------------------------------------
    def step(self, x, y, keep=False):
        """keep: hold on to this step's loss and logits for dump_outputs (only asked of the last timed step)."""
        torch = self.torch
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if self.is_image:
                logits = self.ddp(x)
                loss = self.loss_fn(logits, y)
            else:
                out = self.ddp(input_ids=x, labels=y)
                loss, logits = out.loss, out.logits
                del out
        if keep:
            self.last_loss, self.last_logits = loss.detach(), logits.detach()
        del logits
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        self.opt.step()
        return loss

    def dump_outputs(self, out_dir, max_elems=1 << 21):
        """What the last timed step handed its caller: loss, logits, the averaged gradients (param.grad, in parameter
        order) and the parameters after the optimizer step, as float32 .npy files.  An array larger than max_elems is
        written as the elements at a sorted sample of positions drawn with a fixed seed from its size, so the same
        positions are taken in every run."""
        import numpy as np

        torch = self.torch
        params = [p for p in self.ddp.parameters() if p.requires_grad]
        arrays = {
            "loss": self.last_loss.float().reshape(1),
            "logits": self.last_logits.float().reshape(-1),
            "grads": torch.cat([p.grad.detach().float().reshape(-1) for p in params]),
            "params": torch.cat([p.detach().float().reshape(-1) for p in params]),
        }
        os.makedirs(out_dir, exist_ok=True)
        for name, t in arrays.items():
            n = t.numel()
            if n > max_elems:
                idx = np.sort(np.random.default_rng(n).choice(n, size=max_elems, replace=False))
                t = t[torch.from_numpy(idx).to(t.device)]
            np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))

    def run_resident(self, steps, warmup):
        """`value`: batch already in HBM."""
        torch = self.torch
        (xh, yh), = synthetic_batches(self.args.model, self.args.batch, self.rank, 1, pinned=False)
        x = xh.to(self.device)
        if self.is_image:
            x = x.contiguous(memory_format=torch.channels_last)
        y = yh.to(self.device)
        for _ in range(warmup):
            self.step(x, y)
        torch.cuda.synchronize()
        nv0 = nvlink_bytes(self.device.index) if (self.rank == 0 and self.world > 1) else None  # before the barrier: see allreduce_points
        self.barrier()
        launches0 = self.comm.launches if self.comm is not None else 0
        prof = getattr(self.ddp, "start_profile", None)
        if prof:
            prof()
        sampler = ClockSampler(self.device.index)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        profiled = bool(os.environ.get("BENCH_CUDA_PROFILER"))  # ncu --profile-from-start off: capture the timed region only
        if profiled:
            torch.cuda.profiler.start()
        keep = bool(self.args.dump_outputs)
        e0.record()
        for i in range(steps):
            loss = self.step(x, y, keep=keep and i == steps - 1)
        e1.record()
        self.barrier()
        if profiled:
            torch.cuda.profiler.stop()
        clocks = sampler.stop()
        elapsed = e0.elapsed_time(e1) * 1e-3
        launches = (self.comm.launches - launches0) if self.comm is not None else 0
        kernel = self.ddp.stop_profile() if prof else None
        nv1 = nvlink_bytes(self.device.index) if (self.rank == 0 and self.world > 1) else None
        return elapsed, float(loss.item()), clocks, launches, kernel, nv0, nv1

    def run_e2e(self, steps, warmup):
        """`e2e`: every step's batch is copied from pinned host memory inside the timed region (double-buffered on
        a copy stream) and the loss is read back to the host."""
        torch = self.torch
        host = synthetic_batches(self.args.model, self.args.batch, self.rank, 2, pinned=True)
        dev = [(torch.empty_like(xh, device=self.device), torch.empty_like(yh, device=self.device)) for xh, yh in host]
        ready = [torch.cuda.Event() for _ in host]
        consumed = [torch.cuda.Event() for _ in host]
        loss_host = torch.zeros(steps + warmup, pin_memory=True)

        def prefetch(i):
            k = i % 2
            with torch.cuda.stream(self.copy_stream):
                self.copy_stream.wait_event(consumed[k])
                dev[k][0].copy_(host[k][0], non_blocking=True)
                dev[k][1].copy_(host[k][1], non_blocking=True)
                ready[k].record(self.copy_stream)

        def one(i):
            k = i % 2
            torch.cuda.current_stream().wait_event(ready[k])
            x = dev[k][0].contiguous(memory_format=torch.channels_last) if self.is_image else dev[k][0].clone()
            y = dev[k][1].clone()
            consumed[k].record()  # the landing buffers may be overwritten by the next prefetch from here on
            loss = self.step(x, y)
            loss_host[i].copy_(loss.detach(), non_blocking=True)

        for k in range(2):
            consumed[k].record()
        total = steps + warmup
        prefetch(0)
        for i in range(warmup):
            prefetch(i + 1)
            one(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(warmup, total):
            if i + 1 < total:
                prefetch(i + 1)
            one(i)
        e1.record()
        self.barrier()
        elapsed = e0.elapsed_time(e1) * 1e-3
        h2d = host[0][0].numel() * host[0][0].element_size() + host[0][1].numel() * host[0][1].element_size()
        return elapsed, h2d, loss_host.element_size(), float(loss_host[-1].item())

    def allreduce_points(self):
        """Second half of BASELINE.json's metric: allreduce bus GB/s (fraction of 900 GB/s/dir) on this arm's data path, for
        fp32 buckets of the model's sizes and 256 MiB.  ours: one fused launch (bf16 wire, 1/W).  reference: the
        bf16_compress_hook sequence (cast, div, ncclAllReduce, copy).  busbw = wire bytes / t * 2(W-1)/W, wire = 2 B/element.
        Rank 0 also reads its GPU's NVLink byte counters (nvidia-smi nvlink -gt d) around each timed loop."""
        torch = self.torch
        sizes_mib = sorted(set(self.bucket_sizes))
        if len(sizes_mib) > 5:  # many equal-sized transformer buckets: smallest, the common size, largest
            sizes_mib = [sizes_mib[0], statistics.median_low(self.bucket_sizes), sizes_mib[-1]]
        sizes_mib = sorted(set(sizes_mib) | {256.0})
        out = []
        stream = torch.cuda.Stream(device=self.device)
        k = 2.0 * (self.world - 1) / self.world
        for mib in sizes_mib:
            n = int(mib * (1 << 20) / 4) // 8 * 8
            bufs = [torch.randn(n, device=self.device) for _ in range(2 if mib >= 64 else 6)]
            iters, warm = (20, 5) if mib >= 64 else (100, 20)
            if self.comm is not None:
                def op(b):
                    self.comm.allreduce_(b, stream=stream)
            else:
                import torch.distributed as dist

                def op(b):
                    c = b.to(torch.bfloat16).div_(self.world)
                    dist.all_reduce(c)
                    b.copy_(c)
            with torch.cuda.stream(stream):
                for i in range(warm):
                    op(bufs[i % len(bufs)])
            stream.synchronize()
            # counters are read OUTSIDE the barrier-bracketed region: nvidia-smi takes ~1 s on rank 0 and the other ranks'
            # kernels would spin on it inside their timed loop (the two barriers add a few hundred bytes of traffic)
            nv0 = nvlink_bytes(self.device.index) if self.rank == 0 else None
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                e0.record(stream)
                for i in range(iters):
                    op(bufs[i % len(bufs)])
                e1.record(stream)
            stream.synchronize()
            algo = self.comm.last_algo if self.comm is not None else None
            self.barrier()
            nv1 = nvlink_bytes(self.device.index) if self.rank == 0 else None
            t = self.max_over_ranks(e0.elapsed_time(e1) * 1e-3 / iters)
            row = {"bucket_mib_fp32": mib, "us": round(t * 1e6, 2), "busbw_gbs": round(2 * n / t * k / 1e9, 1),
                   "frac_of_900": round(2 * n / t * k / 1e9 / 900.0, 4)}
            if algo is not None:
                row["algo"] = algo
            if nv0 and nv1:
                row["nvlink_tx_bytes_per_op"] = int((nv1[0] - nv0[0]) / iters)
                row["nvlink_rx_bytes_per_op"] = int((nv1[1] - nv0[1]) / iters)
                row["wire_bytes_S"] = 2 * n
            out.append(row)
            del bufs
        return out

    def parity_check(self):
        """(N>1, our arm) One seeded bucket of each of the model's bucket sizes through comm.allreduce_ with every
        algorithm AUTO can pick, compared on rank 0 against the CPU oracle (the checker, never the product): bit for bit
        for the rank-order kernels; for NVLS (the switch chooses the fp32 summation order) bit for bit wherever the sum is
        order-independent and within one bf16 ulp of the exact sum elsewhere.  Big buckets are checked on windows (head,
        tail, slice boundaries) - the reduction is elementwise."""
        import numpy as np

        import oracle

        torch, W = self.torch, self.world
        algos = ["auto", "oneshot", "twoshot", "twoshot_ll", "twoshot_pipe"] + (["nvls"] if self.comm.has_multicast else [])
        sizes = sorted(set(self.bucket_sizes))
        if len(sizes) > 5:
            sizes = [sizes[0], statistics.median_low(self.bucket_sizes), sizes[-1]]
        res = {"checked_elements": 0, "buckets_mib": sizes, "algos": algos, "bit_exact": True, "auto_picks": {}, "nvls": None, "mismatches": []}
        nvls_stats = {"elements": 0, "differ_from_rank_order": 0, "worse_than_one_bf16_ulp": 0}
        for mib in sizes:
            n = int(mib * (1 << 20) / 4)
            mine = np.random.default_rng(1234 + self.rank).standard_normal(n, dtype=np.float32)
            if n <= (8 << 20):
                wins = [(0, n)]
            else:
                L = 1 << 20
                Ls = ((n + 7) // 8 + W - 1) // W * 8  # elements per rank slice
                starts = {0, n - L, max(0, Ls - L // 2), max(0, (W - 1) * Ls - L // 2), (n // 2) // 8 * 8 + 3}
                wins = [(max(0, min(a, n - L)), max(0, min(a, n - L)) + L) for a in sorted(starts)]
            want = None
            if self.rank == 0:
                full = [mine] + [np.random.default_rng(1234 + r).standard_normal(n, dtype=np.float32) for r in range(1, W)]
                want = [oracle.allreduce(oracle.B2O_F32_WIRE_BF16, [f[a:b] for f in full], 1.0 / W) for a, b in wins]
                exact = [np.sum([oracle.compress(oracle.B2O_F32_WIRE_BF16, f[a:b], 1.0 / W).astype(np.float64) for f in full], axis=0) for a, b in wins]
                del full
            for algo in algos:
                if algo == "oneshot" and mib > 32:
                    continue
                t = torch.from_numpy(mine).to(self.device)
                self.comm.allreduce_(t, algo=algo)
                torch.cuda.synchronize()
                self.comm.check()
                picked = self.comm.last_algo
                if algo == "auto":
                    res["auto_picks"][str(mib)] = picked
                if self.rank != 0:
                    continue
                got = t.cpu().numpy()
                for (a, b), w, ex in zip(wins, want, exact):
                    g = got[a:b]
                    diff = np.flatnonzero((g.view(np.uint32) != w.view(np.uint32)) & ~(np.isnan(g) & np.isnan(w)))
                    res["checked_elements"] += int(b - a)
                    if picked == "nvls":
                        nvls_stats["elements"] += int(b - a)
                        nvls_stats["differ_from_rank_order"] += int(diff.size)
                        if diff.size:
                            ulp = np.maximum(np.abs(ex[diff]), 2.0 ** -126) * 2.0 ** -7
                            nvls_stats["worse_than_one_bf16_ulp"] += int(np.sum(np.abs(g[diff].astype(np.float64) - ex[diff]) > ulp))
                    elif diff.size:
                        res["bit_exact"] = False
                        res["mismatches"].append({"mib": mib, "algo": algo, "picked": picked, "count": int(diff.size), "first": int(a + diff[0])})
            del mine
        if self.comm.has_multicast:
            res["nvls"] = nvls_stats
            if nvls_stats["worse_than_one_bf16_ulp"]:
                res["bit_exact"] = False
        res["vs_nccl_bf16_bit_equal"] = self.nccl_bit_equal(sizes)
        if W == 2 and isinstance(res["vs_nccl_bf16_bit_equal"], dict):
            res["vs_nccl_bf16_w2_bit_equal"] = all(res["vs_nccl_bf16_bit_equal"].values())
        res["note"] = ("bit_exact: every rank-order algorithm (one-shot, two-shot, LL two-shot, pipelined two-shot, and whatever AUTO picked "
                       "among them) equals the CPU oracle bit for bit.  nvls: the NVSwitch's own arithmetic - within one bf16 ulp of the exact "
                       "sum, bit-identical to NCCL's NVLS allreduce (profiles/r02_nvls_rounding.md).  vs_nccl_bf16_bit_equal: AUTO's result "
                       "against the reference hook sequence over NCCL per bucket size - must hold at W=2 (one add); at W>2 it holds "
                       "where both sides take the NVLS path and cannot hold where NCCL uses its ring/tree order with bf16 partial sums.")
        return res

    def nccl_bit_equal(self, sizes_mib):
        """AUTO's result against the reference hook sequence over NCCL (cast, div, ncclAllReduce, copy), bit for bit, per bucket
        size.  torch.distributed is initialised here, after every timed region, for this comparison alone."""
        torch = self.torch
        import torch.distributed as dist

        try:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
                os.environ["NCCL_DEBUG"] = "WARN"
            dist.init_process_group("nccl", rank=self.rank, world_size=self.world, device_id=self.device)
            out = {}
            for mib in sizes_mib:
                n = int(mib * (1 << 20) / 4)
                g = torch.Generator(device=self.device).manual_seed(1234 + self.rank)
                buf = torch.randn(n, device=self.device, generator=g)
                ours = buf.clone()
                self.comm.allreduce_(ours)
                c = buf.to(torch.bfloat16).div_(self.world)
                dist.all_reduce(c)
                ref = buf.clone().copy_(c)
                torch.cuda.synchronize()
                eq = torch.tensor([int(torch.equal(ours, ref))], device=self.device)
                dist.all_reduce(eq, op=dist.ReduceOp.MIN)
                out[f"{mib}:{self.comm.last_algo}"] = bool(eq.item())
                del buf, ours, c, ref
            dist.destroy_process_group()
            return out
        except Exception as e:  # noqa: BLE001 - a missing NCCL must not take the bench line down
            return f"unavailable: {type(e).__name__}: {e}"[:200]

    def close(self):
        if self.comm is not None:
            self.comm.close()
        else:
            import torch.distributed as dist

            if dist.is_initialized():
                dist.destroy_process_group()


def cpu_baseline(world: int, batch: int, bucket_numels, model: str = "resnet50", unit: str = "images"):
    """The oracle (CPU port of the bucket averaging, oracle/allreduce_oracle.c) timed on the host: one pass over
    the model's real buckets for `world` ranks, single thread.  A reported baseline, not a target."""
    import numpy as np

    import oracle

    rng = np.random.default_rng(0)
    n_total = int(sum(bucket_numels))
    w = max(world, 1)
    ins = [[rng.standard_normal(n, dtype=np.float32) for n in bucket_numels] for _ in range(w)]
    t0 = time.perf_counter()
    reps = 0
    while True:
        for b in range(len(bucket_numels)):
            oracle.allreduce(oracle.B2O_F32_WIRE_BF16, [ins[r][b] for r in range(w)], 1.0 / w)
        reps += 1
        if time.perf_counter() - t0 > 10.0 or reps >= 20:
            break
    dt = (time.perf_counter() - t0) / reps
    return {
        "value": round(batch * w / dt, 1),
        "unit": f"{unit}/sec if a step were only the CPU gradient averaging (B*W {unit} per averaging pass)",
        "cores": 1,
        "kind": "port",
        "sample": f"{reps} passes over {model}'s {len(bucket_numels)} gradient buckets ({n_total} fp32 elements) x {w} ranks, "
                  f"oracle/allreduce_oracle.c single-threaded; {round(8 * n_total / dt / 1e9, 2)} GB/s algorithmic",
        "host_cpus": os.cpu_count(),
    }


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus if "RANK" in os.environ else 1)))
    local_rank = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world != args.gpus and rank == 0:
        print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    if args.dump_outputs:
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")  # reproducible cuBLAS; read when its first handle is made
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback for the product path")

    spec = MODELS[args.model]
    if args.batch <= 0:
        args.batch = spec["batch"]
    unit = spec["unit"] + "/sec"
    tr = Trainer(args, rank, world, local_rank)
    elapsed, last_loss, clocks, launches, kernel, nv0, nv1 = tr.run_resident(args.steps, args.warmup)
    elapsed = tr.max_over_ranks(elapsed)
    if args.dump_outputs and rank == 0:  # before run_e2e trains on
        tr.dump_outputs(args.dump_outputs)
    samples = args.batch * world * args.steps
    n_grad = int(sum(p.numel() for p in tr.ddp.parameters() if p.requires_grad))
    line = {
        "metric": spec["metric"],
        "value": round(samples / elapsed, 1),
        "unit": unit,
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": round(elapsed / args.steps * 1e3, 3),
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "bf16",
        "data": "synthetic",
        "impl": args.impl,
        "config": {
            "workload": spec["workload"] % args.batch,
            "global_batch": args.batch * world,
            "parallelism": f"dp{world}",
            "precision": "bf16 autocast compute, fp32 master weights and gradient buckets, %s on the wire" % args.wire,
            "l2": "inputs larger than L2: the batch's activations plus %.1f MiB of fp32 gradient buckets per step exceed the 126 MB L2" % (n_grad * 4 / (1 << 20)),
            "gradient_buckets_mib": tr.bucket_sizes,
        },
        "clocks": clocks,
        "gpu_launches": launches,
        "last_loss": round(last_loss, 4),
    }
    if args.dump_outputs:
        line["deterministic_algorithms"] = "outputs dumped: cuDNN autotuning off, so this is not the headline timing"
    if args.impl == "reference_tuned":
        line["tuned"] = "gradient_as_bucket_view=True, static_graph=True (attribution arm; the headline reference arm uses DDP's defaults)"
    if not args.no_e2e:
        e_elapsed, h2d, d2h, _ = tr.run_e2e(args.steps, args.warmup)
        e_elapsed = tr.max_over_ranks(e_elapsed)
        line["e2e"] = {"value": round(samples / e_elapsed, 1), "unit": unit, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "ms_per_step": round(e_elapsed / args.steps * 1e3, 3)}
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    if os.path.exists(peaks_path):
        try:
            peak = float(json.load(open(peaks_path))["hbm_gbs"])
            peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    if kernel is not None and kernel["launches"]:
        hbm_gbs = kernel["alg_bytes"] / kernel["seconds"] / 1e9
        common = {
            "kernel": kernel["name"], "launches_timed": kernel["launches"], "avg_us": round(kernel["seconds"] / kernel["launches"] * 1e6, 2),
            "per_bucket_us": kernel.get("per_bucket_us"), "alg_bytes_per_launch": kernel["alg_bytes"] // kernel["launches"],
            "gathered_buckets": getattr(tr.ddp, "gathered_buckets", None), "copied_in_buckets": getattr(tr.ddp, "copied_in_buckets", None),
        }
        if world == 1:
            line["roofline"] = {
                "bound": "hbm", "achieved": round(hbm_gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(hbm_gbs / peak, 4), "traffic": None,
                "peak_source": peak_src,
                "note": "8 B per gradient element (read fp32 once, write fp32 once), timed with CUDA events on the comm stream while backward runs beside it; "
                        "with gathered_buckets > 0 this one launch also IS the bucket fill (it reads the per-parameter gradient tensors through the "
                        "segment table): the Reducer-style copy-in pass of round 1 - another 8 B per element and one multi-tensor launch per bucket - no longer exists",
                **common}
            tpath = os.path.join(ROOT, "profiles", "r01_local_pass_traffic.json")
            if os.path.exists(tpath):
                t = json.load(open(tpath))
                # per launch, like `achieved`: scaled from the profiled 30 MiB launch to this run's mean bucket
                per_launch = line["roofline"]["alg_bytes_per_launch"]
                line["roofline"]["traffic"] = int((t["dram_bytes_read"] + t["dram_bytes_write"]) * per_launch / t["alg_bytes"])
                line["roofline"]["traffic_source"] = t["source"] + "; " + t["note"]
        else:
            # the path is NVLink-bound for W >= 2 (DESIGN.md 2.3): algorithmic wire bytes per launch = 2 B/element, reported as
            # nccl-tests bus bandwidth  S/t * 2(W-1)/W  against the 900 GB/s/dir nominal link rate
            k = 2.0 * (world - 1) / world
            busbw = kernel["alg_bytes"] / 4 / kernel["seconds"] * k / 1e9
            traffic = None
            if nv0 and nv1:  # hardware NVLink byte counters of GPU 0 over the timed region (tx + rx), per bucket launch
                traffic = int(((nv1[0] - nv0[0]) + (nv1[1] - nv0[1])) / max(kernel["launches"], 1))
            line["roofline"] = {
                "bound": "nvlink", "achieved": round(busbw, 1), "peak": 900.0, "unit": "GB/s", "frac": round(busbw / 900.0, 4), "traffic": traffic,
                "traffic_source": "nvidia-smi nvlink -gt d on GPU 0 around the timed region: NVLink bytes sent + received per bucket launch "
                                  "(algorithmic wire bytes S = alg_bytes_per_launch / 4; P2P two-shot moves 2(W-1)/W*S each way, NVLS (1+1/W)*S)",
                "peak_source": "nominal NVLink 5 rate per direction per GPU (B200_PROFILING.md; measured peer copy 770 GB/s)",
                "hbm_achieved_gbs": round(hbm_gbs, 1), "hbm_peak_gbs": peak, "hbm_frac": round(hbm_gbs / peak, 4),
                "note": "bus bandwidth of the fused bucket allreduce inside the training step (CUDA events on the comm stream while backward runs beside it)",
                **common}
    if args.sweep and world > 1:
        line["allreduce"] = tr.allreduce_points()
    if args.impl == "b200" and world > 1 and args.parity:
        line["parity"] = tr.parity_check()
    if args.impl != "b200":
        line["cpu_baseline"] = {"value": line["value"], "unit": unit, "cores": os.cpu_count(), "kind": "reference",
                                "sample": "stock torch DistributedDataParallel + NCCL (bf16_compress_hook) - the path `torchx run -s local_cwd dist.ddp` "
                                          "workers execute; launcher and agents on the host cores, gradients on the GPUs"}
        line.setdefault("e2e", {"value": line["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    elif rank == 0 and world == 1 and not args.no_cpu_baseline:
        nums = [int(m * (1 << 20) / 4) for m in (line["config"]["gradient_buckets_mib"] or [97.5])]
        line["cpu_baseline"] = cpu_baseline(world, args.batch, nums, args.model, spec["unit"])
    tr.close()
    if rank == 0:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
