#!/usr/bin/env python
"""Headline benchmark: encrypted-FedAvg rounds on N B200 clients (BASELINE.json).

A *step* is one federated round of the reference's notebook cell 3 (N:233-272) for the medical
CNN (FLPyfhelin.py:118-136): every client (one per GPU) runs ``local_epochs`` x
``steps_per_epoch`` training steps at batch 32 on 256x256x3 images plus the validation passes,
then the round's encrypted FedAvg: CKKS encode + encrypt (n=4096, 3 RNS primes, 109
ciphertexts), ciphertext all-reduce across clients, decrypt + decode, install the average.

Prints ONE JSON line (see the task contract). ``value`` = client-rounds per second summed over
all GPUs (weak scaling: per-GPU work is fixed, one client per GPU); the reference's published
run is 2 client-rounds in 6583.64 s on an unnamed CPU (BASELINE.md).

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nproc-per-node 8 ... bench.py --gpus 8 --steps 5 --warmup 3
  python bench.py --impl reference    # the unmodified reference, if it can be installed
  python bench.py --impl baseline     # same pipeline on NCCL + cuDNN/cuBLAS (the bar to beat)
  python bench.py --dump-outputs DIR  # also write the last timed round's results as DIR/<name>.npy

Inputs are seeded (synthetic data, model init, key pair and encryption randomness), so runs with the same
arguments see identical inputs and two builds can be compared through their --dump-outputs files.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

REF_CLIENT_ROUNDS_PER_SEC = 2.0 / 6583.64   # BASELINE.md: 1 round, 2 clients, 6583.64 s
DUMP_MODEL_MAX = 1 << 22                     # float32 values of the global model written by --dump-outputs (16 MB)


def round_outputs(run):
    """What a caller of ``run_round`` receives from the last round, as float arrays: the averaged global model
    that was decrypted and installed (a fixed, seeded sample of DUMP_MODEL_MAX values when it is larger) and the
    round record's training loss and accuracy."""
    import numpy as np
    import torch

    flat = run.pack.flat.detach().float()
    if flat.numel() > DUMP_MODEL_MAX:
        pick = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MODEL_MAX]
        flat = flat[pick.sort().values.to(flat.device)]
    rec = run.history[-1]
    return {"global_model": flat.cpu().numpy().astype(np.float32),
            "loss": np.array([rec["loss"]], dtype=np.float64),
            "accuracy": np.array([rec["accuracy"]], dtype=np.float64)}


def reference_arm(args):
    """Run the UNMODIFIED reference from baseline/_ref through its own API, if importable."""
    why = None
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    try:
        import importlib.util

        missing = [m for m in ("tensorflow", "Pyfhel", "kerastuner") if importlib.util.find_spec(m) is None]
        if missing:
            why = ("reference needs " + ", ".join(missing) + " (FLPyfhelin.py:3-27); not installed and not in "
                   "/opt/wheelhouse; the reference has no setup.py/pyproject so pip cannot install it either")
        elif not os.path.exists(os.path.join(ref_dir, "FLPyfhelin.py")):
            why = "baseline/_ref/FLPyfhelin.py missing"
    except Exception as e:  # noqa: BLE001
        why = f"probe failed: {e}"
    if why is None:
        why = "reference importable but no dataset folders image/Train, image/Test offline"
    print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "baseline"])
    ap.add_argument("--model", default="medcnn")
    ap.add_argument("--he-preset", default="n4096_l3")
    ap.add_argument("--local-epochs", type=int, default=10)
    ap.add_argument("--steps-per-epoch", type=int, default=23)
    ap.add_argument("--val-steps", type=int, default=3)
    ap.add_argument("--nn-backend", default="auto")
    ap.add_argument("--transport", default=None)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--no-own-baseline", action="store_true",
                    help="skip the NCCL + cuDNN arm that the ours arm also times and reports as own_baseline")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp8"],
                    help="fp8: e4m3 1x1 convolutions for the ResNets (BASELINE configs[4]); the headline config is bf16")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed rounds, write what the last one computed (global model, loss, accuracy) "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        return reference_arm(args)

    # stdout carries exactly ONE line (the result JSON of rank 0): anything a library prints to fd 1
    # meanwhile (e.g. "NCCL version ..." when NCCL_DEBUG is set on the box) is routed to stderr
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    from hefl_b200 import _ext
    from hefl_b200.config import FLConfig
    from hefl_b200.fl import FederatedRunner
    from hefl_b200.fl.data import ResidentFeeder
    from hefl_b200.utils import ClockSampler

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        os.write(result_fd, (json.dumps({"error": "bench.py needs a CUDA device"}) + "\n").encode())
        return 1
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    ops = _ext.ops()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n_rounds, run_round):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        s.record()
        for _ in range(n_rounds):
            run_round()
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e)
        wall = time.perf_counter() - t0
        barrier()
        if world > 1:
            t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        return ms, wall

    def measure(impl, steps, warmup, with_clocks, with_outputs=False):
        """Both passes (end to end, then device-only) of one implementation: "ours" (tcgen05 engine + fused
        ciphertext all-reduce) or "baseline" (the same pipeline on cuDNN/cuBLAS + NCCL all-reduce + mod kernel).
        ``with_outputs``: also return, on the host, what the last device-only round computed."""
        nn_backend = args.nn_backend
        if impl == "baseline":
            nn_backend = "cudnn"
        elif nn_backend == "auto":
            try:
                from hefl_b200.ops import conv_engine  # noqa: F401

                nn_backend = "tcgen05"       # medcnn: the fused engine; ResNets: tcgen05 GEMM convolutions
            except Exception:  # noqa: BLE001
                nn_backend = "cudnn"
        transport = "nccl" if impl == "baseline" else (args.transport or "fused")
        cfg = FLConfig(model=args.model, he_preset=args.he_preset, local_epochs=args.local_epochs,
                       steps_per_epoch=args.steps_per_epoch, val_steps=args.val_steps, clients=world,
                       nn_backend=nn_backend, transport=transport, device="cuda", dtype=args.dtype,
                       deterministic_crypto=True)
        if args.model.startswith("resnet"):
            cfg.image_size, cfg.num_classes = 224, 1000
        run = FederatedRunner(cfg, rank=rank, world=world, device=device)

        def one_round():
            run.run_round(check=False)

        res = {"cfg": cfg, "run": run}
        # ---- pass 1: end to end through the public API (H2D of every step's inputs, D2H of losses)
        h2d = run.train_feed.bytes_per_step
        if not args.skip_e2e:
            for _ in range(warmup):
                one_round()
            l0 = int(ops.launch_count()) + run.trainer.replayed_launches
            e2e_ms, _ = timed(steps, one_round)
            steps_round = cfg.local_epochs * (cfg.steps_per_epoch + cfg.val_steps)
            res["e2e"] = {"value": world * steps / (e2e_ms / 1e3), "unit": "client-rounds/s",
                          "ms_per_round": e2e_ms / steps,
                          "h2d_bytes_per_step": h2d * steps_round, "d2h_bytes_per_step": 8 * steps_round,
                          "h2d_bytes_per_train_step": h2d, "d2h_bytes_per_train_step": 8,
                          "gpu_launches": int(ops.launch_count()) + run.trainer.replayed_launches - l0}
        # ---- correctness of the collective on this box, outside every timed region: the fused kernel's result
        # must equal ncclAllReduce(int64, sum) + mod-q kernel bit for bit on every rank
        if impl == "ours" and world > 1 and run.transport.name == "fused":
            ct = run.encrypt_update()
            snap = ct.data.clone()
            fused = run.aggregate(ct).data.clone()
            dist.all_reduce(snap, op=dist.ReduceOp.SUM)
            ops.reduce_mod_(snap, run.ctx.L, run.ctx.consts)
            ok = torch.tensor([1 if torch.equal(fused, snap) else 0], device=device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            run.transport.check_status()
            run.timer.resolve()
            res["allreduce_checked"] = bool(int(ok))
            if not res["allreduce_checked"]:
                raise RuntimeError("fused ciphertext all-reduce != NCCL all-reduce + mod kernel")
            del snap, fused
        # ---- pass 2: device-only (shard resident in HBM, larger than L2)
        per = len(run.dataset)
        nval = cfg.val_steps * cfg.batch_size
        run.train_feed = ResidentFeeder(run.dataset, range(nval, per), cfg.batch_size, device, seed=rank)
        run.val_feed = ResidentFeeder(run.dataset, range(0, nval), cfg.batch_size, device, seed=rank) if nval else None
        for _ in range(warmup):
            one_round()
        l0 = int(ops.launch_count()) + run.trainer.replayed_launches
        sampler = ClockSampler(local_rank).start() if with_clocks else None
        dev_ms, dev_wall = timed(steps, one_round)
        res["clocks"] = sampler.stop() if sampler else None
        res["launches"] = int(ops.launch_count()) + run.trainer.replayed_launches - l0
        res["stage"] = run.history[-1]["stage_ms"]
        res["dev_ms"], res["dev_wall"] = dev_ms, dev_wall
        res["value"] = world * steps / (dev_ms / 1e3)
        res["shard_mb"] = (per - nval) * cfg.image_size * cfg.image_size * cfg.in_channels / 1e6
        if with_outputs:
            res["outputs"] = round_outputs(run)
        return res

    m = measure(args.impl, args.steps, args.warmup, True, with_outputs=args.dump_outputs is not None)
    cfg, run = m["cfg"], m["run"]
    own_baseline = None
    if args.impl == "ours" and not args.no_own_baseline:
        # The same-box bar (the reference itself cannot run offline): identical pipeline, NCCL all-reduce + mod-q
        # kernel for the ciphertexts, cuDNN/cuBLAS under bf16 autocast + CUDA graphs for the CNN. Same K and W.
        del m["run"]
        run_keep = dict(n=run.ctx.n, L=run.ctx.L, primes=[p.bit_length() for p in run.ctx.primes], n_ct=run.n_ct,
                        ct_numel=run.ct_numel, tname=run.transport.name, algo=getattr(run.transport, "last_algo", None))
        del run
        torch.cuda.empty_cache()
        b = measure("baseline", args.steps, args.warmup, False)
        own_baseline = {"value": b["value"], "unit": "client-rounds/s", "ms_per_step": b["dev_ms"] / args.steps,
                        "nn_backend": b["cfg"].nn_backend, "transport": b["run"].transport.name,
                        "stage_ms_last_round": b["stage"], "gpu_launches": b["launches"]}
        if "e2e" in b:
            own_baseline["e2e"] = {"value": b["e2e"]["value"], "ms_per_round": b["e2e"]["ms_per_round"]}
        del b
    else:
        run_keep = dict(n=run.ctx.n, L=run.ctx.L, primes=[p.bit_length() for p in run.ctx.primes], n_ct=run.n_ct,
                        ct_numel=run.ct_numel, tname=run.transport.name, algo=getattr(run.transport, "last_algo", None))

    if rank == 0:
        value, dev_ms = m["value"], m["dev_ms"]
        out = {
            "metric": "encrypted_fedavg_client_rounds_per_sec", "value": value, "unit": "client-rounds/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": value / REF_CLIENT_ROUNDS_PER_SEC, "dtype": cfg.dtype, "data": "synthetic",
            "impl": args.impl,
            "rounds_per_sec": args.steps / (dev_ms / 1e3), "sec_per_round": dev_ms / 1e3 / args.steps,
            "config": {"model": cfg.model, "global_batch": cfg.batch_size * world, "seq_len": None,
                       "image": [cfg.image_size, cfg.image_size, cfg.in_channels],
                       "parallelism": f"fed-dp{world} (one client per GPU)",
                       "clients": world, "local_epochs": cfg.local_epochs,
                       "train_steps_per_round": cfg.local_epochs * cfg.steps_per_epoch,
                       "val_steps_per_round": cfg.local_epochs * cfg.val_steps,
                       "he": {"scheme": "CKKS", "n": run_keep["n"], "rns_primes": run_keep["L"],
                              "prime_bits": run_keep["primes"],
                              "ciphertexts": run_keep["n_ct"], "ct_bytes_per_client": run_keep["ct_numel"] * 8,
                              "packing": cfg.packing},
                       "nn_backend": cfg.nn_backend, "transport": run_keep["tname"],
                       "allreduce_algo": run_keep["algo"],
                       "key_holder": cfg.key_holder if world > 1 else None,
                       "l2_policy": f"inputs larger than L2: per-client shard {m['shard_mb']:.0f} MB resident in HBM, "
                                    "batches gathered by shuffled index each step"},
            "stage_ms_last_round": m["stage"],
            "clocks": m["clocks"], "gpu_launches": m["launches"], "wall_s": m["dev_wall"],
        }
        if "allreduce_checked" in m:
            out["allreduce_checked"] = m["allreduce_checked"]
        if "e2e" in m:
            out["e2e"] = m["e2e"]
        if own_baseline is not None:
            out["own_baseline"] = own_baseline
            out["vs_own_baseline"] = value / own_baseline["value"]
        if args.dump_outputs is not None:
            import numpy as np

            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in m["outputs"].items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        os.write(result_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
