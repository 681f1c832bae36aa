#!/usr/bin/env python
"""Headline benchmark: LM1B words/sec (default) or ResNet-50 images/sec.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 \
        --master-addr 127.0.0.1 --master-port 29500 bench.py --gpus 8 ...

Config = the reference's (BASELINE.md): LM1B vocab 793 470, emb 512, LSTM
2048→512, 20 steps, batch 128/GPU, sampled softmax 8192, Adagrad, HYBRID sync;
synthetic ids (`lm1b_distributed_driver.py:81-84`), random-init weights.
words/s = steps × batch × num_steps × N / time (`:101-102`).

Timing: W warm-up steps, then exactly K steps bracketed by barrier +
cuda.synchronize, CUDA events on the launching stream, MAX over ranks.  The
embedding / softmax tables (1.6 GB each, + Adagrad slots) are ≫ the 126 MB L2
and every step touches fresh random rows, so no explicit L2 flush is needed
("inputs larger than L2").  `e2e` times the same K steps through the public
API (`sess.run`) with per-step H2D of the batch from pinned memory and a D2H
read of the loss.

`--dump-outputs DIR` writes what the last timed step returned (loss and final LSTM
state for LM1B) as .npy files: the inputs and weights are seeded, so two builds run with
the same arguments can be compared output for output.  The benchmark writes nothing into
the source tree, which may be read-only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True        # no __pycache__ in a possibly read-only tree
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BASELINE_LM1B_WPS = 277000.0     # Parallax-HYBRID, 48× TITAN Xp (BASELINE.md)
BASELINE_RESNET_IPS = 7550.0     # Parallax-HYBRID, 48× TITAN Xp (BASELINE.md)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="parallax_b200",
                    choices=["parallax_b200", "reference", "nccl"])
    ap.add_argument("--model", default="lm1b", choices=["lm1b", "resnet50", "ncf", "bert"])
    ap.add_argument("--run-option", default="HYBRID")
    ap.add_argument("--dtype", default="bf16")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--small", action="store_true",
                    help="tiny config for plumbing checks (NOT a valid number)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dense-nvls", default="auto", choices=["auto", "on", "off"],
                    help="NVLS multicast dense step: auto = on a full 8-GPU box")
    ap.add_argument("--protocol", default="nvlink", choices=["nvlink", "nccl"],
                    help="nccl = same engine / same CUDA graph, every cross-GPU byte through "
                         "NCCL collectives (the in-engine library baseline)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the secondary blocks (same-engine NCCL arm, fp32 LM1B, "
                         "ResNet-50, sustained run, self-check)")
    ap.add_argument("--comm", action="store_true",
                    help="with --no-extras: still report the graph-replayed comm probes")
    ap.add_argument("--sustained-s", type=float, default=3.0,
                    help="length of the additional sustained-clock run (seconds)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned "
                         "(rank 0) as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out, path, limit=DUMP_LIMIT_BYTES):
    """Write the arrays of one step's result as `path/<name>.npy`.  Floating arrays are
    stored as float32 (float64 stays float64), integer and boolean ones as float64.  The
    files stay under `limit` bytes in all: the budget is shared out smallest array first,
    and an array larger than its share is replaced by the elements of its flattened form at
    sorted indices drawn with a fixed seed, so every run samples the same positions.
    Returns {name: {"shape": original shape, "stored": elements written}}."""
    import re
    import numpy as np
    import torch
    arrays = {}
    for name, v in out.items():
        if torch.is_tensor(v):
            v = v.detach()
            v = v.float() if v.is_floating_point() and v.dtype != torch.float64 else v.double()
            arrays[name] = v.cpu().numpy()
        elif isinstance(v, (bool, int, float)):
            arrays[name] = np.asarray(v, dtype=np.float64)
    os.makedirs(path, exist_ok=True)
    left, written = limit, {}
    for i, name in enumerate(sorted(arrays, key=lambda k: (arrays[k].nbytes, k))):
        a = arrays[name]
        shape = list(a.shape)
        share = left // (len(arrays) - i) - 1024          # room for the .npy header
        if a.nbytes > share:
            n = max(share // a.itemsize, 0)
            idx = np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))
            a = a.reshape(-1)[idx]
        fn = os.path.join(path, re.sub(r"[^A-Za-z0-9_.-]", "_", name) + ".npy")
        np.save(fn, a)
        left -= os.path.getsize(fn)
        written[name] = {"shape": shape, "stored": int(a.size)}
    return written


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region.

    The query process is started before the warm-up so it is already streaming when
    the timed region begins (its start-up alone can exceed a short timed region);
    every line is stamped on arrival and `stop(t0, t1)` reports the samples that fall
    inside the timed window (median SM clock under load)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index=0, period_ms=50):
        self.proc, self.lines, self.gpu, self.period_ms = None, [], gpu_index, period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-i", str(self.gpu), "-lms", str(self.period_ms)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    @classmethod
    def _parse(cls, stamped):
        out = []
        for ts, ln in stamped:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                rec = (ts, float(f[1]), float(f[2]), float(f[3]))
            except ValueError:
                continue
            out.append(rec + ([nm for nm, v in zip(cls.NAMES, f[5:9])
                               if v.lower().startswith("active")],))
        return out

    def stop(self, t0=None, t1=None):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        return self.window(t0, t1)

    def window(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        recs = self._parse(list(self.lines))
        inside = [r for r in recs if (t0 is None or r[0] >= t0) and (t1 is None or r[0] <= t1)]
        window = "timed region"
        if not inside:
            # a very short timed region can fall between two samples: use the samples
            # taken under the same load just before it (the warm-up steps)
            inside, window = ([r for r in recs if t1 is None or r[0] <= t1][-5:] or recs), \
                "last warm-up samples (timed region shorter than the sampling period)"
        sm = sorted(r[1] for r in inside)
        reasons = sorted({nm for r in inside for nm in r[4]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": max((r[2] for r in inside), default=None),
                "power_w_max": max((r[3] for r in inside), default=None),
                "samples": len(inside), "samples_total": len(recs), "window": window,
                "period_ms": self.period_ms, "reasons": reasons}


def reference_arm(args):
    """Reference arm: the UNMODIFIED reference from baseline/_ref through its
    own public API.  Its pure-python `parallax` package installs offline
    (pip --no-deps from a /tmp copy, see DESIGN.md) but importing it needs the
    snuspl TensorFlow r1.11 fork + Horovod 0.16.3 + mpirun, none of which exist
    for CUDA 12.9 / sm_100 or in /opt/wheelhouse — so the arm reports
    `unavailable` with the actual import error."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    env = dict(os.environ, PYTHONPATH=ref_dir)
    why = "baseline/_ref is empty (reference not installed)"
    if os.path.isdir(os.path.join(ref_dir, "parallax")):
        r = subprocess.run([sys.executable, "-c", "import parallax"], env=env,
                           cwd="/tmp", capture_output=True, text=True)
        if r.returncode == 0:
            why = ("reference imports, but its runtime (TF1.11 fork kernels built for "
                   "compute_35/70, Horovod, mpirun) cannot run on sm_100")
        else:
            last = (r.stderr.strip().splitlines() or ["import failed"])[-1]
            why = ("reference `import parallax` fails: %s; it requires the snuspl "
                   "TensorFlow r1.11 fork + Horovod 0.16.3 + mpirun (not in "
                   "/opt/wheelhouse, no sm_100 build)" % last)
    if int(os.environ.get("RANK", "0")) == 0:     # one line per job under torchrun
        print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


def build_lm1b(args, parallax, torch):
    from parallax_b200.models.lm1b import LM1B, lm1b_graph
    if args.small:
        kw = dict(vocab_size=50000, emb_size=128, state_size=512, projected_size=128,
                  num_sampled=1024, num_steps=8, num_shards=8)
        batch = args.batch or 32
    else:
        kw = dict(vocab_size=793470, emb_size=512, state_size=2048, projected_size=512,
                  num_sampled=8192, num_steps=20, num_shards=32)
        batch = args.batch or 128
    model = LM1B(lazy=True, **kw)
    graph = lm1b_graph(model, batch_size=batch)
    T, V = kw["num_steps"], kw["vocab_size"]

    def make_batch(gen):
        x = torch.randint(0, V, (batch, T), generator=gen, dtype=torch.int64)
        y = torch.randint(0, V, (batch, T), generator=gen, dtype=torch.int64)
        return {"x": x, "y": y}
    desc = {"model": "lm1b(vocab=%d,emb=%d,lstm=%d->%d,steps=%d,sampled=%d)" % (
        V, kw["emb_size"], kw["state_size"], kw["projected_size"], T, kw["num_sampled"]),
        "per_gpu_batch": batch, "seq_len": T, "optimizer": "adagrad(0.2)",
        "items_per_step": batch * T}
    return graph, make_batch, desc, "lm1b_words_per_sec", "words/s", BASELINE_LM1B_WPS


def build_resnet(args, parallax, torch):
    from parallax_b200.models.resnet import resnet50, resnet_graph
    batch = args.batch or (8 if args.small else 64)
    model = resnet50(num_classes=1000)
    graph = resnet_graph(model)
    hw = 64 if args.small else 224

    def make_batch(gen):
        return {"images": torch.randn(batch, 3, hw, hw, generator=gen),
                "labels": torch.randint(0, 1000, (batch,), generator=gen)}
    desc = {"model": "resnet50_v1", "per_gpu_batch": batch, "seq_len": hw,
            "optimizer": "momentum(0.9)", "items_per_step": batch}
    return graph, make_batch, desc, "resnet50_images_per_sec", "images/s", BASELINE_RESNET_IPS


def build_ncf(args, parallax, torch):
    from parallax_b200.models.ncf import NeuMF, ncf_graph
    users = 1_000_000 if args.small else 100_000_000
    items = 100_000 if args.small else 1_000_000
    batch = args.batch or (4096 if args.small else 65536)
    model = NeuMF(users, items, num_partitions=8, lazy=True)
    graph = ncf_graph(model)

    def make_batch(gen):
        return {"users": torch.randint(0, users, (batch,), generator=gen),
                "items": torch.randint(0, items, (batch,), generator=gen),
                "labels": torch.randint(0, 2, (batch,), generator=gen)}
    desc = {"model": "neumf(users=%d,items=%d,row=32+32 fp32)" % (users, items),
            "per_gpu_batch": batch, "seq_len": 1, "optimizer": "adam(1e-3, lazy sparse)",
            "items_per_step": batch}
    return graph, make_batch, desc, "ncf_samples_per_sec", "samples/s", None


def build_bert(args, parallax, torch):
    from parallax_b200.models.bert import Bert, bert_graph
    if args.small:
        model, batch, T = Bert(hidden=256, layers=4, heads=4, ff=1024), args.batch or 8, 128
    else:
        model, batch, T = Bert(), args.batch or 16, 512
    graph = bert_graph(model)
    nm = max(1, int(T * 0.15))

    def make_batch(gen):
        return {"input_ids": torch.randint(0, 30522, (batch, T), generator=gen),
                "mlm_positions": torch.randint(0, T, (batch, nm), generator=gen),
                "mlm_labels": torch.randint(0, 30522, (batch, nm), generator=gen)}
    desc = {"model": "bert_large" if not args.small else "bert_small", "per_gpu_batch": batch,
            "seq_len": T, "optimizer": "adam(1e-4)+clip(1.0)", "items_per_step": batch * T}
    return graph, make_batch, desc, "bert_tokens_per_sec", "tokens/s", None


def _max_over_ranks(torch, dist, world, dev, vals):
    t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]


def measure(args, model, dtype, K, Wm, world, rank, protocol="nvlink", e2e=True,
            comm_stamps=False, sustained_s=0.0, sampler=None, dump_dir=None):
    """Build a session for `model`, run Wm warm-up + exactly K timed steps (device events,
    max over ranks) and the optional extra regions; returns the result block.  With
    `dump_dir`, rank 0 writes the last timed step's result there before any later step
    runs (a replayed CUDA graph returns the same tensors every step)."""
    import torch
    import torch.distributed as dist
    import parallax_b200 as parallax
    from parallax_b200.parallel import nvops
    margs = argparse.Namespace(**vars(args))
    margs.model, margs.dtype = model, dtype
    builder = {"lm1b": build_lm1b, "resnet50": build_resnet, "ncf": build_ncf,
               "bert": build_bert}[model]
    graph, make_batch, desc, metric, unit, baseline = builder(margs, parallax, torch)
    sc = {"compute_dtype": dtype, "cuda_graph": not args.no_graph}
    if args.dense_nvls != "auto":
        sc["dense_nvls"] = args.dense_nvls == "on"
    run_option = "MPI" if model == "resnet50" else args.run_option
    cfg = parallax.Config(run_option=run_option, search_partitions=False, sess_config=sc)
    if protocol == "nccl":
        cfg.communication_config = parallax.CommunicationConfig(
            parallax.PSConfig(protocol="nccl"))
    sess, nw, wid, _ = parallax.parallel_run(graph, "localhost:0", sync=True,
                                             parallax_config=cfg)
    eng = sess.engine
    dev = eng.comm.device
    gen = torch.Generator().manual_seed(99 + rank)
    if sc["cuda_graph"]:
        Wm = max(Wm, int(sc.get("graph_warmup", 3)) + 2)
    items = desc["items_per_step"] * world

    # ---- device-timed arm: inputs resident on the device -------------------
    batches = [{k: v.to(dev) for k, v in make_batch(gen).items()} for _ in range(4)]
    for i in range(Wm):
        eng.train_step(batches[i % 4])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_w0 = time.time()
    l0 = nvops.launches["n"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(K):
        out = eng.train_step(batches[i % 4])
    e1.record()
    torch.cuda.synchronize()
    t_w1 = time.time()
    launches = nvops.launches["n"] - l0
    if world > 1:
        dist.barrier()
    ms, = _max_over_ranks(torch, dist, world, dev, [e0.elapsed_time(e1)])
    res = {"metric": metric, "value": items * K / (ms / 1e3), "unit": unit,
           "ms_per_step": ms / K, "steps": K, "warmup": Wm, "dtype": dtype,
           "gpu_launches": launches, "loss": float(out["loss"]),
           "cuda_graph": bool(getattr(eng, "graph_captured", False)),
           "run_option": eng.run_option.lower(), "protocol": protocol,
           "_desc": desc, "_baseline": baseline, "_window": (t_w0, t_w1)}
    if dump_dir is not None and rank == 0:
        res["dump_outputs"] = {"dir": dump_dir, "arrays": dump_outputs(out, dump_dir)}

    # ---- sustained run: the same step for >= sustained_s seconds -------------
    if sustained_s > 0:
        n_s = max(K, int(sustained_s * 1e3 / max(ms / K, 1e-3)) + 1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        s_w0 = time.time()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(n_s):
            eng.train_step(batches[i % 4])
        s1.record()
        torch.cuda.synchronize()
        s_w1 = time.time()
        if world > 1:
            dist.barrier()
        ms_s, = _max_over_ranks(torch, dist, world, dev, [s0.elapsed_time(s1)])
        res["sustained"] = {"steps": n_s, "seconds": ms_s / 1e3, "ms_per_step": ms_s / n_s,
                            "value": items * n_s / (ms_s / 1e3), "unit": unit}
        if sampler is not None and rank == 0:
            res["sustained"]["clocks"] = sampler.window(s_w0, s_w1)

    # ---- end-to-end arm: public API, pinned H2D in, loss D2H out -------------
    if e2e:
        host_batches = [{k: v.pin_memory() for k, v in make_batch(gen).items()}
                        for _ in range(4)]
        h2d = sum(v.numel() * v.element_size() for v in host_batches[0].values())
        for i in range(3):
            sess.run(["loss", "train_op"], {k: [v] for k, v in host_batches[i % 4].items()})
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(K):
            loss, _ = sess.run(["loss", "train_op"],
                               {k: [v] for k, v in host_batches[i % 4].items()})
        s1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms2, = _max_over_ranks(torch, dist, world, dev, [s0.elapsed_time(s1)])
        res["e2e"] = {"value": items * K / (ms2 / 1e3), "unit": unit,
                      "ms_per_step": ms2 / K, "h2d_bytes_per_step": h2d,
                      "d2h_bytes_per_step": 4, "last_loss": float(loss[0])}

    # ---- exposed communication, measured inside the CUDA-graph replay ---------
    if comm_stamps:
        try:
            bd = eng.comm_breakdown_replayed(batches[0], steps=20)
            keys = sorted(k for k in bd if k != "graph_replay")
            vals = _max_over_ranks(torch, dist, world, dev, [bd[k] for k in keys])
            res["comm"] = {k: round(v, 4) for k, v in zip(keys, vals)}
            res["comm"]["how"] = ("%globaltimer probes captured in the step graph, 20 replays, "
                                  "max over ranks" if bd["graph_replay"] else "eager steps")
        except Exception as e:  # pragma: no cover
            res["comm"] = {"error": repr(e)}
    sess.close()
    return res


def _public(block, keep=("value", "unit", "ms_per_step", "steps", "warmup", "dtype", "loss",
                         "e2e", "sustained", "comm", "gpu_launches", "cuda_graph",
                         "protocol", "run_option", "metric")):
    return {k: block[k] for k in keep if k in block}


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)
    import torch
    import torch.distributed as dist
    if args.impl == "nccl":
        from baseline.nccl_reference import main as nccl_main
        return nccl_main(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    assert world == args.gpus or world == 1, "launch with torchrun for --gpus > 1"
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device", "metric": "lm1b_words_per_sec"}))
        return 1
    from parallax_b200.parallel.fabric import Comm
    comm = Comm.from_env()            # one process group for every arm below
    torch.manual_seed(1234 + rank)
    K, Wm = args.steps, max(args.warmup, 3)
    extras = not args.no_extras and not args.small
    sampler = ClockSampler(comm.device.index or 0)
    if rank == 0:
        sampler.start()          # streaming by the time the timed region starts

    # ---- correctness first: the live fabric vs a single-device oracle ---------
    selfcheck = None
    if extras:
        from parallax_b200.utils import selfcheck as sc_
        try:
            r = sc_.check(world, rank, "HYBRID", "adagrad", steps=4, resource="localhost:0")
            oks = comm.all_gather_object((r["ok"], r["max_abs_err"]))
            selfcheck = {"ok": all(o for o, _ in oks), "max_abs_err": max(e for _, e in oks),
                         "what": "MLP+embedding, HYBRID/adagrad, 4 steps vs single-device "
                                 "oracle on the concatenated batch", "backend": r["backend"]}
        except Exception as e:
            selfcheck = {"ok": False, "error": repr(e)}
        if not selfcheck["ok"]:
            if rank == 0:
                print(json.dumps({"error": "self-check failed", "selfcheck": selfcheck,
                                  "metric": "lm1b_words_per_sec"}))
            return 1

    main_blk = measure(args, args.model, args.dtype, K, Wm, world, rank,
                       protocol=args.protocol, e2e=not args.no_e2e,
                       comm_stamps=extras or args.comm,
                       sustained_s=args.sustained_s if extras else 0.0, sampler=sampler,
                       dump_dir=args.dump_outputs)
    clocks = sampler.window(*main_blk["_window"]) if rank == 0 else None
    blocks = {}
    if extras and args.model == "lm1b":
        def arm(name, **kw):
            try:
                blocks[name] = _public(measure(args, **kw))
            except Exception as e:      # a secondary block must never lose the headline
                blocks[name] = {"error": repr(e)}
        if world > 1 and args.protocol == "nvlink":
            arm("same_engine_nccl", model="lm1b", dtype=args.dtype, K=K, Wm=Wm, world=world,
                rank=rank, protocol="nccl", e2e=False)
            b = blocks["same_engine_nccl"]
            if "value" in b:
                b["what"] = ("identical model, engine and CUDA-graph capture; dense = "
                             "ncclAllReduce on the bucket + local fused optimizer, sparse = "
                             "ncclAllGather of (ids, rows) + owner apply, lookup = "
                             "ncclAllGather(ids) + local gather + ncclReduceScatter")
                b["nvlink_over_nccl"] = main_blk["value"] / b["value"]
        arm("lm1b_fp32", model="lm1b", dtype="fp32", K=K, Wm=Wm, world=world, rank=rank,
            e2e=False)
        arm("resnet50", model="resnet50", dtype="bf16", K=K, Wm=Wm, world=world, rank=rank,
            e2e=True)
        if "value" in blocks.get("resnet50", {}):
            blocks["resnet50"]["vs_baseline"] = blocks["resnet50"]["value"] / BASELINE_RESNET_IPS
            blocks["resnet50"]["config"] = {"model": "resnet50_v1", "global_batch": 64 * world,
                                            "parallelism": "dp%d/mpi(AR)/sync" % world,
                                            "optimizer": "momentum(0.9)", "layout": "channels_last"}
    sampler.stop()
    desc, baseline = main_blk["_desc"], main_blk["_baseline"]
    if rank == 0:
        rec = {
            "metric": main_blk["metric"], "value": main_blk["value"], "unit": main_blk["unit"],
            "n_gpus": world, "steps": K, "warmup": main_blk["warmup"],
            "ms_per_step": main_blk["ms_per_step"],
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (main_blk["value"] / baseline) if baseline else None,
            "dtype": args.dtype,
            "data": "synthetic (random ids / images, random-init weights)",
            "impl": "parallax_b200",
            "config": {"model": desc["model"],
                       "global_batch": desc["per_gpu_batch"] * world,
                       "seq_len": desc["seq_len"],
                       "parallelism": "dp%d/%s/sync" % (world, main_blk["run_option"]),
                       "optimizer": desc["optimizer"], "protocol": args.protocol,
                       "l2": "inputs larger than L2 (tables >> 126 MB, fresh random rows each step)"
                       if args.model == "lm1b" else "activations+weights >> L2 per step",
                       "cuda_graph": main_blk["cuda_graph"], "valid": not args.small},
            "baseline": {"value": baseline,
                         "what": "Parallax-HYBRID on 48x TITAN Xp (BASELINE.md)"},
            "clocks": clocks, "e2e": main_blk.get("e2e"),
            "gpu_launches": main_blk["gpu_launches"], "comm": main_blk.get("comm"),
            "sustained": main_blk.get("sustained"), "loss": main_blk["loss"],
            "selfcheck": selfcheck,
        }
        if "dump_outputs" in main_blk:
            rec["dump_outputs"] = main_blk["dump_outputs"]
        rec.update(blocks)
        print(json.dumps(rec))
    comm.shutdown()
    return 0


if __name__ == "__main__":
    sys.exit(main())
