"""Single configuration object for the engine (SURVEY.md §5.6).

The reference has no config system: module globals (FLPyfhelin.py:31-36), literals
(``p=65537`` :332, callbacks :186-187) and hard-coded paths. Here everything lives in one
dataclass that can be overridden from the CLI (``--key value``) or the environment
(``HEFL_KEY=value``) and is echoed into every result record.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
from dataclasses import dataclass, field
from typing import Any, Optional, Sequence

# SEAL-style upper bounds on log2(Q) for 128/192/256-bit security (ternary secret).
SEC_MAX_LOGQ = {
    128: {1024: 27, 2048: 54, 4096: 109, 8192: 218, 16384: 438, 32768: 881},
    192: {1024: 19, 2048: 37, 4096: 75, 8192: 152, 16384: 305, 32768: 611},
    256: {1024: 14, 2048: 29, 4096: 58, 8192: 118, 16384: 237, 32768: 476},
}

# Named HE parameter sets used by BASELINE.json configs.
HE_PRESETS = {
    # configs[1]: medical CNN, n=4096, 3 RNS primes (36+36+37 = 109 bits)
    "n4096_l3": dict(n=4096, prime_bits=(36, 36, 37), scale_bits=40),
    # configs[2]: ResNet-18, n=8192, 4 primes (<= 218 bits)
    "n8192_l4": dict(n=8192, prime_bits=(54, 54, 54, 55), scale_bits=40),
    # configs[4]: ResNet-50, n=16384, 8 primes (<= 438 bits)
    "n16384_l8": dict(n=16384, prime_bits=(54,) * 8, scale_bits=40),
    "n16384_l4": dict(n=16384, prime_bits=(54,) * 4, scale_bits=40),
    # CPU plumbing config
    "n2048_l1": dict(n=2048, prime_bits=(54,), scale_bits=40),
}


@dataclass
class FLConfig:
    # model / data
    model: str = "medcnn"            # medcnn | cnn2 | resnet18 | resnet50
    image_size: int = 256             # reference: 256x256x3 (FLPyfhelin.py:35)
    in_channels: int = 3
    num_classes: int = 2
    batch_size: int = 32              # FLPyfhelin.py:33
    local_epochs: int = 10            # notebook N:30
    steps_per_epoch: int = 23         # 720 training images / 32 (notebook log N:120)
    val_steps: int = 3                # 80 validation images / 32
    lr: float = 1e-3                  # FLPyfhelin.py:31
    lr_decay: float = 1e-4            # FLPyfhelin.py:140 (INIT_LR / 10)
    dtype: str = "bf16"               # compute dtype of local training
    nn_backend: str = "tcgen05"       # tcgen05 (hand-written kernels) | cudnn (baseline)
    # federation
    clients: int = 2
    rounds: int = 1
    compat_sequential_clients: bool = False   # reproduce quirk Q1 (FLPyfhelin.py:180-193)
    key_holder: int = 0                       # rank that GENERATES the key pair (OS entropy), is the only one to keep the
                                              # secret key, owns no chunk of the fused all-reduce (never loads a peer's
                                              # un-aggregated ciphertext), decrypts the aggregate and broadcasts the averaged
                                              # model -- the reference's roles: aggregation with get_pk (FLPyfhelin.py:370),
                                              # get_sk only in decrypt (:284). -1: rank 0 generates and hands sk to every
                                              # rank (every client can decrypt; weaker, kept for experiments)
    deterministic_crypto: bool = False        # tests / debugging ONLY: derive the key pair and every encryption seed from
                                              # ``seed`` (public!) instead of OS entropy, so runs are bit-reproducible;
                                              # bench.py sets it (synthetic data, reproducible inputs), never for real data
    pairwise_masks: bool = False              # add PRG masks (X25519-agreed pair seeds, +/- per pair) to each client's
                                              # ciphertext before the all-reduce; they cancel in the sum
    allow_dropouts: bool = False              # clients may sit a round out (participation mask): K becomes a runtime
                                              # value agreed by a 1-element all-reduce and folded into the decode scale
    debug_precision: bool = False             # also all-reduce the PLAINTEXT updates and record the CKKS error of the
                                              # round (debug only: it defeats the privacy the ciphertext path provides)
    debug_poison: bool = False                # overwrite ciphertext / scratch buffers with a poison pattern between rounds
    # HE
    he_preset: str = "n4096_l3"
    packing: str = "slots"            # slots (canonical embedding, N/2 per ct) | coeff (N per ct)
    sec: int = 128
    transport: str = "fused"          # fused | nccl | loopback
    allreduce_algo: str = "auto"      # auto | one_shot | two_shot | multimem
    # misc
    seed: int = 1234
    device: str = "cuda"
    workdir: str = "."
    log_jsonl: Optional[str] = None
    timeout_s: float = 120.0          # bounded waits on device flags / collectives

    def he_params(self) -> dict:
        return dict(HE_PRESETS[self.he_preset])

    def to_json(self) -> str:
        return json.dumps(dataclasses.asdict(self), sort_keys=True)

    @classmethod
    def from_args(cls, argv: Optional[Sequence[str]] = None, **defaults: Any) -> "FLConfig":
        """Build a config from defaults < environment (HEFL_*) < CLI flags."""
        cfg = cls(**defaults)
        for f in dataclasses.fields(cls):
            env = os.environ.get("HEFL_" + f.name.upper())
            if env is not None:
                setattr(cfg, f.name, _coerce(env, f.type, getattr(cfg, f.name)))
        p = argparse.ArgumentParser(add_help=False)
        for f in dataclasses.fields(cls):
            p.add_argument("--" + f.name.replace("_", "-"), dest=f.name, default=None)
        ns, _ = p.parse_known_args(argv)
        for f in dataclasses.fields(cls):
            v = getattr(ns, f.name)
            if v is not None:
                setattr(cfg, f.name, _coerce(v, f.type, getattr(cfg, f.name)))
        return cfg


def _coerce(text: str, typ: Any, current: Any) -> Any:
    if isinstance(current, bool):
        return str(text).lower() in ("1", "true", "yes", "on")
    if isinstance(current, int):
        return int(text)
    if isinstance(current, float):
        return float(text)
    if current is None:
        return None if text in ("", "None", "none") else text
    return text
