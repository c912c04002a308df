"""bench.py -- CODAE hot path on B200: train samples/s (headline) + candidate scores/s, with roofline and CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload polyvore|embedding|modanet] [--dtype fp32|bf16|fp32_simt]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   (one rank per GPU, NCCL)
  python bench.py --impl reference ...   the reference's own CPU implementation of the same step on the host cores (the
                                          unmodified reference classes from baseline/_ref; the oracle port if that is absent)
  python bench.py ... --dump-outputs DIR  also writes what the last timed step computed as DIR/*.npy (same arguments, same
                                          inputs: two builds can be compared output for output)

Default workload: the polyvore-shaped multi-slot step (BASELINE.json configs[3]: 10 x Linear(4096, 4096), B = 8192 per GPU,
bf16 tensor-core engine) -- the largest single-GPU training configuration and the one the tensor-pipe bar is written for.
The shipped small-batch configs (embedding.yaml at fp32 -- the reference's precision, on the fp32-parity tensor-core engine --
AND bf16, the modanet yaml at bf16) and the 10 M-row scoring sweep are measured in the same run and reported as secondary
blocks of the same JSON line (`secondary`, `scoring`); each small-batch block also carries `epoch_mode`: the scripts' loop for
a resident dataset (FusedStep.train_epoch: sampler on the device, 32 steps per CUDA-graph launch, wall clock around an epoch).

A "step" is one pass of the training-step hot path over one batch of synthetic embeddings of the config's shape
(corrupt -> encoder/decoder GEMMs -> loss -> backward GEMMs -> [all-reduce] -> clip -> Adam).  `value` is the
whole-job samples/s with the dataset resident in HBM (timed with CUDA events, max over ranks); `e2e` is the same
metric through the public API (codae.tool.FusedStep.step(staged=...)) with the batch rows coming from pinned host
memory every step and the loss read back every step.  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "mui-deepautoencoder_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (yaml, S, E, z, nin, nout, B per GPU, k_max, lr, wd, clip, default dtype, N observations)
    "embedding": dict(yaml="config/embedding.yaml", S=3, E=512, z=1536, nin=4, nout=4, B=128, k_max=1, lr=1e-5, wd=1e-4,
                      clip=True, dtype="bf16", N=131072, seed=27493045),
    "modanet": dict(yaml="config/modanet_merge_top_bottom_shoe.yaml", S=3, E=512, z=1536, nin=3, nout=3, B=32, k_max=1,
                    lr=1e-4, wd=1e-2, clip=False, dtype="bf16", N=131072, seed=50493213),
    "polyvore": dict(yaml="config/polyvore_multislot.yaml", S=8, E=512, z=4096, nin=4, nout=4, B=8192, k_max=2, lr=1e-4,
                     wd=1e-2, clip=True, dtype="bf16", N=1048576, seed=50493213, cpu_B=2048),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops"], tensor_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def layer_dims(w):
    from codae.model import EmbeddingDenoisingAutoencoder  # noqa: F401
    io = w["S"] * w["E"]
    inc_in, inc_out = (io - w["z"]) // w["nin"], (io - w["z"]) // w["nout"]
    dims = [(io, io)]
    last = None
    for i in range(1, w["nin"]):
        a, last = max(io - (i - 1) * inc_in, w["z"]), max(io - i * inc_in, w["z"])
        dims.append((a, last))
    dims.append((last, w["z"]))
    for i in range(w["nout"]):
        a, last = min(w["z"] + i * inc_out, io), min(w["z"] + (i + 1) * inc_out, io)
        dims.append((a, last))
    dims.append((last, io))
    return dims


def synthetic_rows(N, io, seed, device):
    """Scaled dataset rows of the config's shape: |N(0,1)| * Bernoulli(0.7), divided by (max - min) like
    ConcatenatedEmbeddingDataset does (reference concatenated_embedding_dataset.py:69-74)."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randn((N, io), generator=g, device=device).abs_()
    x *= (torch.rand((N, io), generator=g, device=device) < 0.7)
    return x / float(x.max() - x.min())


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own classes (baseline/_ref) or, without them, the oracle port, on the host cores
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference(w, steps, warmup, seed=0):
    """One CPU step = the reference's loop body over a bounded sample of the workload: cpu_B rows (the config's batch for the
    small-batch configs, 2048 rows of the 8192-row polyvore batch).  kind "reference": the unmodified reference classes
    (baseline/live_reference.py); kind "port": oracle/codae_oracle.py."""
    io, B = w["S"] * w["E"], w.get("cpu_B", w["B"])
    dims = layer_dims(w)
    n = max(4 * B, 1024)
    data = synthetic_rows(n, io, seed, "cpu")
    shape = "%d x Linear(%d, %d)" % (len(dims), dims[0][0], dims[0][1])
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import live_reference as LR
    if LR.available() and os.environ.get("CODAE_CPU_ARM", "reference") != "port":
        r = LR.train_steps(w, data, B, steps, warmup, seed)
        dt, cores, kind = r["seconds"], r["cores"], "reference"
        what = "the unmodified reference classes (baseline/_ref) driven by the reference's loop body"
    else:
        from oracle import codae_oracle as O
        torch.manual_seed(seed)
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        relu = [True] * len(dims)
        relu[w["nin"]] = False
        relu[-1] = False
        W = [torch.empty(o, i).uniform_(-1, 1) * (6.0 / (i + o)) ** 0.5 for i, o in dims]
        b = [torch.zeros(o) for _, o in dims]
        dae = O.OracleDAE(W, b, relu, w["lr"], w["wd"], w["clip"])
        arch = [dict(size=w["E"], position=p) for p in range(0, io, w["E"])]
        bm, nmiss, _ = O.binary_masks(arch, w["k_max"])
        import random
        random.seed(seed)
        tbl = O.mask_table_compat(n, bm.shape[0])
        rng = np.random.RandomState(seed)
        t0 = None
        for s in range(warmup + steps):
            if s == warmup:
                t0 = time.perf_counter()
            idx = rng.randint(0, n, size=B).tolist()
            _, fmask = O.get_masks(bm, nmiss, tbl, idx, 0, w["k_max"])       # the reference's per-sample Python loop
            dae.step_embedding(data[idx], fmask)
        dt, kind = time.perf_counter() - t0, "port"
        what = "the oracle port of the reference step"
    return dict(value=B * steps / dt, unit="samples/s", cores=cores, kind=kind,
                sample="%d steps of %d rows%s (%s) with %s on %d host threads"
                       % (steps, B, "" if B == w["B"] else " (of the %d-row batch)" % w["B"], shape, what, cores),
                ms_per_step=1e3 * dt / steps)


def cpu_scoring(E, rows=1_000_000):
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import live_reference as LR
    r = LR.scoring_sweeps(E, rows)            # the reference's op (metering.py:67-69) is a torch call: same code either way
    return r["scores"] / r["seconds"]


def workload_config(name, w, dims, world):
    io = w["S"] * w["E"]
    P = sum(i * o + o for i, o in dims)
    big = "larger than the 126 MB L2"
    return {"workload": "%s (%s): %d x Linear, io=%d, B=%d/GPU, k_max=%d, N=%d" % (name, w["yaml"], len(dims), io, w["B"], w["k_max"], w["N"]),
            "params": P, "l2_policy": "no flush: every step streams weights + Adam state (%.0f MB), activations and random dataset "
                                      "rows, %s" % (32.0 * P / 1e6, big),
            "parallelism": "dp%d" % world}


# ----------------------------------------------------------------------------------------------------------------
def train_block(name, dtype, K, Wm, args, env, e2e=True, dump_dir=None):
    """One training workload on this rank's GPU: device-timed `value`, end-to-end `e2e`, per-kernel rooflines; with dump_dir,
    what the last timed step computed (dump_outputs)."""
    import torch.distributed as dist
    from codae import _C
    from codae.dataset import ConcatenatedEmbeddingDataset
    from codae.model import EmbeddingDenoisingAutoencoder
    from codae.tool import Corrupter, FusedStep
    rank, world, dev, local = env["rank"], env["world"], env["dev"], env["local"]
    w = dict(WORKLOADS[name])
    io, B = w["S"] * w["E"], w["B"]
    dims = layer_dims(w)
    torch.manual_seed(w["seed"])
    data = synthetic_rows(w["N"], io, w["seed"], dev)
    ds = ConcatenatedEmbeddingDataset.__new__(ConcatenatedEmbeddingDataset)
    ds.data, ds.nb_observation, ds.embedding_size, ds.nb_used_category = data, w["N"], w["E"], w["S"]
    ds.arch = [dict(name=str(i), size=w["E"], type="regression", position=i * w["E"]) for i in range(w["S"])]
    model = EmbeddingDenoisingAutoencoder(io, w["z"], w["E"], w["nin"], w["nout"], False)
    assert model.dims == dims
    model.set_compute_dtype(dtype)
    model.to(dev)
    cor = Corrupter(w["N"], ds.arch, w["k_max"], dev, seed=w["seed"])
    fs = FusedStep(model, cor, data, lr=w["lr"], weight_decay=w["wd"], clip=w["clip"], world_size=world,
                   use_graph=not args.no_graph, wgrad_sqnorm=False if args.no_wgrad_sqnorm else None,
                   dp_mode=args.dp_mode)
    rng = np.random.RandomState(w["seed"] + rank)
    batches = torch.from_numpy(rng.randint(0, w["N"], size=(Wm + K, B))).to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: `value` ---------------------------------------------------------------------
    for s in range(Wm):
        fs.step(batches[s], global_batch=B * world)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(Wm, Wm + K):
        fs.step(batches[s], global_batch=B * world)
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    clocks = sampler.stop() if sampler else None
    launches = K * fs.kernel_launches
    loss_last = fs.last_loss(B)
    if dump_dir:
        fs.flush()                # data-parallel peer mode gathers the master-weight shards: every rank takes part
        if rank == 0:
            dump_outputs(dump_dir, fs, B, loss_last)
    out = {"metric": "train samples/s", "value": world * B * K / (ms / 1e3), "unit": "samples/s", "n_gpus": world, "steps": K,
           "warmup": Wm, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16" if fs_dtype(dtype, model) == "bf16" else "f32", "data": "synthetic",
           "config": workload_config(name, w, dims, world), "engine": engine_name(model), "dp_mode": fs.dp_mode,
           "loss_last_step": loss_last, "clocks": clocks, "gpu_launches": launches, "cuda_graph": not args.no_graph}

    # ---- end-to-end through the public API with host buffers: `e2e` -------------------------------------------------
    if e2e:
        table = cor.device_tables()[0]
        host_rows = torch.empty((4, B, io), dtype=torch.float32).pin_memory()
        host_tab = torch.empty((4, B, table.shape[1]), dtype=torch.int16).pin_memory()
        for j in range(4):
            host_rows[j].copy_(data[batches[j]].cpu())
            host_tab[j].copy_(table[batches[j]].cpu())
        # two staging buffers: the host->device copy of step s+1 (copy stream) overlaps the kernels of step s; every step's
        # copy and every step's loss read-back are inside the timed region
        st_rows = [torch.empty((B, io), dtype=torch.float32, device=dev) for _ in range(2)]
        st_tab = [torch.empty((B, table.shape[1]), dtype=torch.int16, device=dev) for _ in range(2)]
        loss_host = torch.zeros(4, dtype=torch.float64).pin_memory()
        Ke = max(10, K // 2)
        copy_stream = torch.cuda.Stream(device=dev)
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]

        def stage(s):
            j = s % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[j])          # the step that last used this buffer has finished
                st_rows[j].copy_(host_rows[s % 4], non_blocking=True)
                st_tab[j].copy_(host_tab[s % 4], non_blocking=True)
                copied[j].record(copy_stream)

        def e2e_loop(n):
            main = torch.cuda.current_stream()
            for j in range(2):
                consumed[j].record(main)
            stage(0)
            last = 0.0
            for s in range(n):
                j = s % 2
                if s + 1 < n:
                    stage(s + 1)
                main.wait_event(copied[j])
                fs.step(None, global_batch=B * world, staged=(st_rows[j], st_tab[j]))
                consumed[j].record(main)
                loss_host.copy_(fs.acc, non_blocking=True)
                main.synchronize()                           # the user sees this step's loss before issuing the next step
                last = float(loss_host[3]) / (B * io)
            main.synchronize()
            return last

        e2e_loop(6)
        barrier()
        t0 = time.perf_counter()
        e2e_loop(Ke)
        barrier()
        e2e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev)
        if world > 1:
            dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
        out["e2e"] = {"value": world * B * Ke / (float(e2e_ms.item()) / 1e3), "unit": "samples/s",
                      "h2d_bytes_per_step": B * io * 4 + B * table.shape[1] * 2, "d2h_bytes_per_step": 32, "steps": Ke,
                      "api": "codae.tool.FusedStep.step(staged=(rows, mask_table_rows))"}
        del host_rows, host_tab, st_rows, st_tab
        if B <= 1024 and world == 1:
            # the scripts' own loop for a RESIDENT dataset (train_dae_on_embedding.py --graph): FusedStep.train_epoch -- permutation
            # drawn on the device, 32 steps per CUDA-graph launch, one monitor read-back per epoch.  Wall clock around whole epochs.
            rows = torch.arange(w["N"], dtype=torch.int64, device=dev)
            gen = torch.Generator(device=dev)
            gen.manual_seed(w["seed"])
            fs.train_epoch(rows[:64 * B], B, generator=gen)             # captures the 32-step graph
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_steps = fs.train_epoch(rows, B, generator=gen)
            mon = fs.read_monitors()                                   # the epoch's one device->host read
            dt_epoch = time.perf_counter() - t0
            out["epoch_mode"] = {"value": n_steps * B / dt_epoch, "unit": "samples/s", "steps": n_steps, "ms_per_step": 1e3 * dt_epoch / n_steps,
                                 "api": "codae.tool.FusedStep.train_epoch (device sampler, 32 steps per graph launch)",
                                 "h2d_bytes_per_step": 0, "d2h_bytes_per_epoch": 32, "rows_seen": mon["rows"]}

    # ---- per-kernel durations inside a real step (CUDA events on the launch stream) -> roofline ----------------------
    prof = profile_step(fs, batches[0], B, world, name)      # every rank: the steps inside contain the collective
    out.update({"roofline": prof["roofline"], "rooflines": prof["rooflines"], "kernels": prof["kernels"], "step_floor": prof["floor"]})
    # whole step against its floor: tensor-bound configs -> GEMM flops at the sustained bf16 peak (+ the HBM-bound kernels at
    # the HBM peak); small-batch configs -> the HBM floor of SURVEY section 8(d)
    fl = prof["floor"]
    out["step_vs_floor"] = {"floor_ms": fl["ms"], "bound": fl["bound"], "frac": fl["ms"] / (ms / K)}
    del fs, model, cor, data, ds, batches
    torch.cuda.empty_cache()
    return out, w


DUMP_MAX_ELEMS = 1 << 22      # per array (16 MB of float32): a dump stays under 64 MB
DUMP_SEED = 20240917


def dump_outputs(out_dir, fs, B, loss):
    """What a caller of FusedStep.step holds after the last timed step, as out_dir/<name>.npy: the loss, the monitor sums, the
    reconstruction of the last batch, the model's parameters and their gradients (weights then bias of every layer, in
    model.dims order).  An array of more than DUMP_MAX_ELEMS elements is replaced by a fixed, seeded sample (rows of the
    reconstruction; positions of the parameter vector, the same for parameters and gradients): the same positions every run,
    so that two builds compare output for output."""
    model = fs.model
    g = torch.Generator().manual_seed(DUMP_SEED)

    y = fs._bufs[B]["acts"][-1][:, :fs.io]
    if y.numel() > DUMP_MAX_ELEMS:
        y = y[torch.randperm(B, generator=g)[:DUMP_MAX_ELEMS // fs.io].sort().values.to(y.device)]
    P = model.nb_parameters()
    pos = None if P <= DUMP_MAX_ELEMS else torch.randint(0, P, (DUMP_MAX_ELEMS,), generator=g).sort().values.to(fs.dev)

    def params(flat):
        v = torch.cat([torch.cat([model.weight_view(flat, l).reshape(-1), model.bias_view(flat, l)]) for l in range(len(model.dims))])
        return (v if pos is None else v[pos]).cpu().numpy()

    arrays = {"loss": np.array([loss], dtype=np.float64),
              "monitors": fs.acc.cpu().numpy(),                    # sums of the full / partial loss, rows, last step's sum
              "reconstruction": y.cpu().numpy(),
              "parameters": params(model.flat),
              "gradients": params(fs.gflat)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def scoring_block(args, env, E, seed, model_for_swaps=None):
    import torch.distributed as dist
    from codae.tool.inference import ComplementarityScorer, shard_rows
    rank, world, dev = env["rank"], env["world"], env["dev"]
    pk = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lo, n_local = shard_rows(args.catalog, world, rank)
    g = torch.Generator(device=dev).manual_seed(seed + 17)
    catalog = torch.rand((n_local, E), generator=g, device=dev)
    q = torch.rand((1, E), generator=g, device=dev)
    reps = 10
    scoring = None
    for tag, cat in (("f32", catalog), ("bf16", None)):
        if cat is None:
            cat = catalog.to(torch.bfloat16)
        sc = ComplementarityScorer(cat, E, metric="sqerr", k=10, row_offset=lo)
        for _ in range(3):
            sc.topk(q)
        barrier()
        e0.record()
        for _ in range(reps):
            sc.topk(q)
        e1.record()
        barrier()
        sms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(sms, op=dist.ReduceOp.MAX)
        sweep_ms = float(sms.item()) / reps
        # kernel alone (local sweep, no merge collective) for the roofline
        e0.record()
        for _ in range(reps):
            sc.topk_local(q)
        e1.record()
        torch.cuda.synchronize()
        k_ms = e0.elapsed_time(e1) / reps
        bytes_per = n_local * E * cat.element_size()
        blk = {"metric": "candidate-outfit scores/s", "value": args.catalog / (sweep_ms / 1e3), "unit": "scores/s",
               "catalog_rows": args.catalog, "E": E, "dtype": tag, "k": 10, "ms_per_sweep": sweep_ms, "scaling": "strong",
               "kernel_ms": k_ms,
               "roofline": {"bound": "hbm", "achieved": bytes_per / (k_ms / 1e3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                            "frac": bytes_per / (k_ms / 1e3) / 1e9 / pk["hbm"], "traffic": measured_traffic("scoring_" + tag, n_local),
                            "kernel": "score_topk_kernel", "peak_source": pk["src"],
                            "algorithmic_per_launch": bytes_per}}
        if scoring is None:
            scoring = blk
        else:
            scoring["bf16_catalog"] = blk
        del sc
    del catalog
    torch.cuda.empty_cache()
    return scoring


def swap_block(args, env, seed):
    """Swaps scored by FULL reconstruction (candidate substituted, whole outfit through the DAE): the GEMM-bound reading of
    "scores candidate item swaps by reconstruction error", on the embedding.yaml model."""
    import torch.distributed as dist
    from codae.model import EmbeddingDenoisingAutoencoder
    from codae.tool.inference import SwapScorer, shard_rows
    rank, world, dev = env["rank"], env["world"], env["dev"]
    w = WORKLOADS["embedding"]
    io = w["S"] * w["E"]
    model = EmbeddingDenoisingAutoencoder(io, w["z"], w["E"], w["nin"], w["nout"], False)
    model.set_compute_dtype("bf16")
    model.to(dev)
    lo, n_local = shard_rows(args.catalog, world, rank)
    n_sw = min(n_local, 1 << 20)
    g = torch.Generator(device=dev).manual_seed(seed + 19)
    catalog = torch.rand((n_sw, w["E"]), generator=g, device=dev)
    sw = SwapScorer(model, catalog, w["E"], k=10, row_offset=lo, chunk=8192)
    outfit = torch.rand(io, generator=g, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        sw.topk(outfit, 1)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        sw.topk(outfit, 1)
    e1.record()
    torch.cuda.synchronize()
    sms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(sms, op=dist.ReduceOp.MAX)
    sw_ms = float(sms.item()) / 3
    sw_flops = 2.0 * sum(i * o for i, o in model.dims) * n_sw
    return {"metric": "candidate swaps/s (full DAE reconstruction per swap)", "value": world * n_sw / (sw_ms / 1e3),
            "unit": "swaps/s", "swaps_per_rank": n_sw, "chunk": 8192, "ms": sw_ms, "engine": "bf16",
            "tflops": sw_flops / (sw_ms / 1e3) / 1e12}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", type=str, default="polyvore", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", type=str, default=None, choices=["fp32", "bf16", "fp32_simt"],
                    help="fp32: the reference's precision on tensor cores (bf16 triples); bf16: 1e-2 mode; fp32_simt: FFMA engine (A/B)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-scoring", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the small-batch configs reported beside the primary workload")
    ap.add_argument("--no-prefetch", action="store_true", help="weight tiles are not requested ahead of the PDL wait")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-pdl", action="store_true", help="A/B: launch without programmatic dependent launch")
    ap.add_argument("--no-splitk", action="store_true", help="A/B: single-pass small-batch contractions")
    ap.add_argument("--no-persistent", action="store_true", help="A/B: one tile per CTA for the large contractions")
    ap.add_argument("--no-wgrad-sqnorm", action="store_true",
                    help="A/B (1 GPU): cooperative norm + Adam kernel instead of sum(dW^2) partials from the weight-gradient kernels")
    ap.add_argument("--no-tma-store", action="store_true", help="A/B: per-thread stores instead of TMA bulk stores (both GEMM kernels)")
    ap.add_argument("--dp-mode", type=str, default=None, choices=["peer", "nccl"],
                    help="data parallel: fused peer-memory reduce-scatter + sharded Adam + all-gather kernel (default) or NCCL all-reduce")
    ap.add_argument("--catalog", type=int, default=10_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, monitors, reconstruction, parameters and "
                         "gradients; larger arrays as a fixed, seeded sample) as DIR/<name>.npy")
    args = ap.parse_args()
    w0 = dict(WORKLOADS[args.workload])
    big = args.workload == "polyvore"
    K = args.steps if args.steps is not None else (30 if big else 2000)
    Wm = args.warmup if args.warmup is not None else (5 if big else 50)
    if Wm < 3 and args.impl == "ours":
        Wm = 3                          # timing rules: at least 3 warm-up steps on the GPU arm
    dtype = args.dtype or w0["dtype"]
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference(w0, K, Wm)
        print(json.dumps({"impl": "reference", "metric": "train samples/s", "value": r["value"], "unit": "samples/s",
                          "n_gpus": args.gpus, "steps": K, "warmup": Wm, "ms_per_step": r["ms_per_step"],
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": workload_config(args.workload, w0, layer_dims(w0), world),
                          "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                          "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)
    from codae import _C
    if args.no_pdl:
        _C.set_option(dev, _C.OPT_PDL, 0)
    if args.no_prefetch:
        _C.set_option(dev, _C.OPT_WEIGHT_PREFETCH, 0)
    if args.no_splitk:
        _C.set_option(dev, _C.OPT_SPLITK, 0)
    if args.no_persistent:
        _C.set_option(dev, _C.OPT_PERSISTENT, 0)
    if args.no_tma_store:
        _C.set_option(dev, _C.OPT_TMA_STORE, 0)
        _C.set_option(dev, _C.OPT_TMA_STORE_PERSISTENT, 0)
    env = dict(rank=rank, world=world, dev=dev, local=local)

    out, w = train_block(args.workload, dtype, K, Wm, args, env, e2e=True, dump_dir=args.dump_outputs)
    # ---- the shipped small-batch configs, each at its stated precision and in the other mode (same run, same box) -------
    if not args.no_secondary and args.workload == "polyvore" and args.dtype is None:
        sec = {}
        for tag, name, dt_ in (("embedding.yaml fp32 (reference precision)", "embedding", "fp32"),
                               ("embedding.yaml bf16", "embedding", "bf16"),
                               ("modanet_merge_top_bottom_shoe.yaml bf16", "modanet", "bf16")):
            try:
                blk, _ = train_block(name, dt_, 500, 30, args, env, e2e=True)
                keep = ("value", "unit", "ms_per_step", "dtype", "engine", "config", "e2e", "epoch_mode", "roofline", "step_vs_floor", "kernels",
                        "gpu_launches", "steps", "warmup", "loss_last_step", "dp_mode")
                sec[tag] = {k: blk[k] for k in keep if k in blk}
            except Exception as ex:      # the primary line is the contract: report, do not lose the run
                sec[tag] = {"error": repr(ex)[:300]}
        out["secondary"] = sec
    if not args.no_scoring:
        out["scoring"] = scoring_block(args, env, w["E"], w["seed"])
        try:
            out["scoring"]["swap_reconstruction"] = swap_block(args, env, w["seed"])
        except Exception as ex:
            out["scoring"]["swap_reconstruction"] = {"error": repr(ex)[:300]}
        if rank == 0 and not args.no_cpu:
            out["scoring"]["cpu_baseline"] = {"value": cpu_scoring(w["E"]), "unit": "scores/s", "cores": os.cpu_count(), "kind": "reference",
                                              "sample": "3 x cosine_similarity + topk over 1M x %d rows (the reference's op, metering.py:67-69)" % w["E"]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if not args.no_cpu:
        r = cpu_reference(w, 4 if big else 200, 1 if big else 3)
        out["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def engine_name(model):
    from codae import _C
    e = model.engine_dtype()
    return {_C.BF16: "tcgen05 bf16 (fp32 accumulate in TMEM)", _C.F32: "exact-fp32 FFMA",
            _C.F32X3: "tcgen05 fp32-parity (bf16 triples hi/mid/lo, 6 MMAs per k-step, fp32 accumulate in TMEM)"}.get(e, str(e))


_TRAFFIC = None


def measured_traffic(key, rows=None):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed `ncu --set full` capture of this
    round (profiles/r02_traffic.json, written by tools/ncu_summary.py --traffic); None when no capture exists for `key`."""
    global _TRAFFIC
    if _TRAFFIC is None:
        path = os.path.join(ROOT, "profiles", "r02_traffic.json")
        _TRAFFIC = json.load(open(path)) if os.path.exists(path) else {}
    v = _TRAFFIC.get(key)
    if v is None:
        return None
    b = v.get("bytes_per_launch")
    if rows is not None and v.get("rows"):
        b = b * rows / v["rows"]          # captured on a smaller catalog: DRAM bytes scale with the rows swept
    return b


def fs_dtype(dtype, model):
    from codae import _C
    return {_C.BF16: "bf16", _C.F32X3: "fp32x3"}.get(model.engine_dtype(), "fp32")


def profile_step(fs, idx, B, world, name):
    """Per-kernel-group durations and rooflines.  One eager step is recorded (which ABI calls, with which arguments);
    every group is then captured R times into one CUDA graph and replayed between ONE CUDA-event pair on the launching
    stream, so a group's time is GPU time of exactly its launches (no host launch gaps).  Rooflines use ALGORITHMIC bytes / flops
    (SURVEY.md section 8d) against the measured peaks."""
    from codae import _C
    pk = peaks()
    model = fs.model
    dims = model.dims
    wrapped = ["corrupt_fwd", "linear_fwd", "mse_loss_fwd_bwd", "linear_wgrad", "linear_dgrad", "grad_sqnorm", "counter_add", "adam_step",
               "clip_adam_step", "linear_wgrad_sq", "adam_step_partials", "dp_adam_step"]
    orig = {n: getattr(_C, n) for n in wrapped}
    calls = {n: [] for n in wrapped}

    def wrap(n):
        def f(*a, **k):
            calls[n].append((a, k))
            return orig[n](*a, **k)
        return f

    saved_graph = fs.use_graph
    fs.use_graph = False
    try:
        for n in wrapped:
            setattr(_C, n, wrap(n))
        fs.step(idx, global_batch=B * world)
    finally:
        for n in wrapped:
            setattr(_C, n, orig[n])
        fs.use_graph = saved_graph
    torch.cuda.synchronize()
    R = 10
    kernels = {}
    for n in wrapped:
        if not calls[n]:
            continue
        for a, k in calls[n]:
            orig[n](*a, **k)
        torch.cuda.synchronize()
        # R repetitions of the group captured into ONE CUDA graph: GPU time without host launch gaps (an eager replay of
        # 10 us kernels through ctypes is host bound)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(R):
                for a, k in calls[n]:
                    orig[n](*a, **k)
        gr.replay()
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        gr.replay()
        s1.record()
        torch.cuda.synchronize()
        ms = s0.elapsed_time(s1) / R
        kernels[n] = {"ms_per_step": ms, "launches_per_step": len(calls[n]), "us_per_launch": 1e3 * ms / len(calls[n])}
        del gr
    step_ms = sum(k["ms_per_step"] for k in kernels.values())
    for k in kernels.values():
        k["share"] = k["ms_per_step"] / step_ms
    Wsum = sum(i * o for i, o in dims)
    W1 = dims[0][0] * dims[0][1]
    P = model.nb_parameters()
    io = dims[0][0]
    act = sum(i + o for i, o in dims)
    bf = fs.eng == _C.BF16
    x3 = fs.eng == _C.F32X3
    tc = bf or x3
    # bytes per GEMM operand element in the engine's own format: bf16 2, fp32 4, fp32 as a bf16 triple 6 (DESIGN.md section 5)
    sw = 2 if bf else (6 if x3 else 4)
    shadow = 2 if bf else (6 if x3 else 0)
    small = B <= 1024      # small batch: a contraction is bound by streaming its weights / writing dW once, not by the tensor pipe
    algo = {  # name: (bound, algorithmic bytes or flops per STEP, unit note)
        "adam_step": ("hbm", (28 + shadow) * P),
        "clip_adam_step": ("hbm", (32 + shadow) * P),
        "adam_step_partials": ("hbm", (28 + shadow) * P),
        "grad_sqnorm": ("hbm", 4 * P),
        "corrupt_fwd": ("hbm", B * io * (4 + sw)),
        "mse_loss_fwd_bwd": ("hbm", B * io * (4 + 4 + sw)),
        "linear_fwd": ("hbm", Wsum * sw + B * act * sw) if small else ("tensor", 2.0 * B * Wsum),
        "linear_dgrad": ("hbm", (Wsum - W1) * sw + B * act * sw) if small else ("tensor", 2.0 * B * (Wsum - W1)),
        "linear_wgrad": ("hbm", Wsum * 4 + B * act * sw) if small else ("tensor", 2.0 * B * Wsum),
    }
    algo["linear_wgrad_sq"] = algo["linear_wgrad"]
    # useful flops against the bf16 tensor peak; the fp32-parity engine issues six bf16 MMAs per fp32 product
    tensor_peak = pk["tensor_sustained"] if bf else (pk["tensor_sustained"] / 6 if x3 else pk["tensor_sustained"] / 2)
    rooflines = {}
    for n, (bound, work) in algo.items():
        if n not in kernels:
            continue
        sec = kernels[n]["ms_per_step"] / 1e3
        if bound == "hbm":
            ach, peak, unit = work / sec / 1e9, pk["hbm"], "GB/s"
        else:
            ach, peak, unit = work / sec / 1e12, tensor_peak, "TFLOP/s"
        rooflines[n] = {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                        "traffic": measured_traffic("%s_%s_%s" % (name, "bf16" if bf else ("fp32x3" if x3 else "fp32"), n)),
                        "kernel": n, "share_of_step": kernels[n]["share"], "peak_source": pk["src"],
                        "algorithmic_per_launch": work / kernels[n]["launches_per_step"]}
    # the dominant KERNEL: the three contractions are one kernel (tc05_gemm_kernel / simt_gemm_kernel)
    gemm = [n for n in ("linear_fwd", "linear_dgrad", "linear_wgrad", "linear_wgrad_sq") if n in kernels]
    gemm_ms = sum(kernels[n]["ms_per_step"] for n in gemm)
    others = {n: kernels[n]["ms_per_step"] for n in rooflines if n not in gemm}
    top_other = max(others, key=others.get)
    if gemm_ms >= others[top_other]:
        work = sum(algo[n][1] for n in gemm)
        bound = algo[gemm[0]][0]
        launches = sum(kernels[n]["launches_per_step"] for n in gemm)
        ach = work / (gemm_ms / 1e3) / (1e9 if bound == "hbm" else 1e12)
        peak = pk["hbm"] if bound == "hbm" else tensor_peak
        roof = {"bound": bound, "achieved": ach, "peak": peak, "unit": "GB/s" if bound == "hbm" else "TFLOP/s", "frac": ach / peak,
                "traffic": None, "kernel": ("tc05_gemm_persistent_kernel (fwd + dgrad + wgrad launches)" if not small else
                                            "tc05_gemm_kernel (fwd + dgrad + wgrad launches)") if bf else
                                           ("tc05_gemm_kernel<BN, 3 planes> (fwd + dgrad + wgrad launches)" if x3 else
                                            "simt_gemm_kernel (fwd + dgrad + wgrad launches)"),
                "share_of_step": gemm_ms / step_ms, "peak_source": pk["src"], "algorithmic_per_launch": work / launches,
                "note": "B <= 1024: bound by streaming the weights once per contraction (weights + activations bytes), not by the "
                        "tensor pipe; latency-bound in practice, see DESIGN.md section 7" if small else
                        ("useful fp32 flops vs 1/6 of the sustained cuBLAS bf16 peak (six bf16 MMAs per fp32 product)" if x3 else
                         "dense bf16 contraction vs the sustained cuBLAS bf16 peak")}
        if bf and bound == "tensor":
            # the same rate against cuBLAS's BURST figure (best single 8192^3 launch; the launches of a step run back to back, so the
            # sustained figure is the denominator of `frac`) and against the nominal dense bf16 peak of the part
            roof["frac_of_burst_peak"] = ach / pk["tensor"]
            roof["frac_of_nominal_2250"] = ach / 2250.0
            if os.environ.get("CODAE_CTA_PAIR", "1") != "0" and "persistent" in roof["kernel"]:
                roof["kernel"] = "tc05_gemm_persistent_kernel<256, CTA pair> (fwd + dgrad + wgrad launches; cta_group::2, 256 x 256 tiles)"
        if x3 and bound == "hbm":
            # the same time against the fp32 information content (4 B per weight / activation element instead of the triple's 6)
            roof["frac_at_fp32_bytes"] = roof["frac"] * 4.0 / 6.0
    else:
        roof = rooflines[top_other]
    # DRAM traffic per launch of the dominant kernel from this round's committed `ncu --set full` capture (profiles/r02_traffic.json)
    roof["traffic"] = measured_traffic("%s_%s_%s" % (name, "bf16" if bf else ("fp32x3" if x3 else "fp32"), "gemm" if "gemm" in roof.get("kernel", "") else roof.get("kernel", "")))
    hbm_bytes = (32 + (4 if x3 else 0)) * P + B * 20 * io
    if small:
        floor_bytes = hbm_bytes + 3 * Wsum * sw
        floor = {"bound": "hbm", "hbm_bytes_per_step": floor_bytes, "ms": floor_bytes / (pk["hbm"] * 1e9) * 1e3, "sum_of_kernel_ms": step_ms}
    else:
        flops = 2.0 * B * (3 * Wsum - W1)
        floor = {"bound": "tensor", "flops_per_step": flops, "hbm_bytes_per_step": hbm_bytes,
                 "ms": flops / (tensor_peak * 1e12) * 1e3 + hbm_bytes / (pk["hbm"] * 1e9) * 1e3,
                 "gemm_ms_at_sustained_peak": flops / (tensor_peak * 1e12) * 1e3, "sum_of_kernel_ms": step_ms}
    return {"kernels": kernels, "roofline": roof, "rooflines": rooflines, "floor": floor}


if __name__ == "__main__":
    main()
