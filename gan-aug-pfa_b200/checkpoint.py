"""Checkpoint / resume for the native trainers (SURVEY.md §8(f) rank 4).

The reference only ever saves `state_dict()`s (train_gan.py:149-153, train.py:307-321): no optimizer state, no step
count, no RNG state, and nothing resumes.  Here a checkpoint holds
  * the model `state_dict()`s in the REFERENCE's format (same keys / shapes / dtypes: `generate_synthetic_data.py:48` and
    `evaluate.py:345` load them unchanged — `export_reference_state_dicts` writes exactly those files), and
  * what a bit-faithful resume needs on top: the Adam / AdamW moments and step counters (flat fp32 buffers in the
    engine's segment layout, with the segment table for validation), the dropout mask counter and seed, and the
    torch CPU / CUDA RNG states (data order, augmentation).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

FORMAT = "gap_b200_checkpoint_v1"


def _net_state(net) -> dict:
    st = net.store
    return {
        "state_dict": {k: v.detach().cpu().clone() for k, v in net.state_dict().items()},
        "adam_m": st.m.detach().cpu().clone(),
        "adam_v": st.v.detach().cpu().clone(),
        "adam_step": int(st.step_dev.item()) if st.step_dev is not None else int(st.step),
        "segments": {k: list(v) for k, v in st.segs.items()},
    }


def _load_net(net, d: dict) -> None:
    if {k: list(v) for k, v in net.store.segs.items()} != d["segments"]:
        raise ValueError("checkpoint was written by an engine with a different parameter layout")
    net.load_state_dict(d["state_dict"])            # also re-packs the bf16 operands
    st = net.store
    with torch.no_grad():
        st.m.copy_(d["adam_m"].to(st.m.device))
        st.v.copy_(d["adam_v"].to(st.v.device))
    st.step = int(d["adam_step"])
    if st.step_dev is not None:
        st.step_dev.fill_(st.step)


def _rng_state(device) -> dict:
    out = {"cpu": torch.get_rng_state()}
    if torch.cuda.is_available() and torch.device(device).type == "cuda":
        out["cuda"] = torch.cuda.get_rng_state(device)
    return out


def _set_rng_state(d: dict, device) -> None:
    torch.set_rng_state(d["cpu"])
    if "cuda" in d and torch.cuda.is_available():
        torch.cuda.set_rng_state(d["cuda"], device)


def trainer_state(trainer, extra: Optional[dict] = None) -> dict:
    """Everything needed to continue a Pix2PixTrainer run as if it had never stopped."""
    torch.cuda.synchronize(trainer.dev)
    return {"format": FORMAT, "kind": "pix2pix", "norm": trainer.norm,
            "channels": {"input_nc": trainer.input_nc, "output_nc": trainer.output_nc},
            "G": _net_state(trainer.G), "D": _net_state(trainer.D),
            "hyper": {"lr_g": trainer.lr_g, "lr_d": trainer.lr_d, "betas": list(trainer.betas)},
            "dropout": {"seed": trainer.G.dropout_seed, "calls": trainer.G.dropout_calls},
            "rng": _rng_state(trainer.dev), "extra": extra or {}}


def load_trainer_state(trainer, state: dict, restore_rng: bool = True) -> dict:
    if state.get("format") != FORMAT or state.get("kind") != "pix2pix":
        raise ValueError("not a gap_b200 pix2pix checkpoint")
    norm = state.get("norm", "batch")       # checkpoints written before InstanceNorm support are BatchNorm runs
    if norm != trainer.norm:
        raise ValueError(f"checkpoint was written by a norm={norm!r} trainer; this trainer uses norm={trainer.norm!r}")
    # checkpoints written before channel counts were recorded are 3 -> 3 runs
    ch = state.get("channels", {"input_nc": 3, "output_nc": 3})
    mine = {"input_nc": trainer.input_nc, "output_nc": trainer.output_nc}
    if ch != mine:
        raise ValueError(f"checkpoint was written by a trainer with input_nc={ch['input_nc']}, output_nc={ch['output_nc']}; "
                         f"this trainer has input_nc={mine['input_nc']}, output_nc={mine['output_nc']}")
    _load_net(trainer.G, state["G"])
    _load_net(trainer.D, state["D"])
    trainer.lr_g, trainer.lr_d = state["hyper"]["lr_g"], state["hyper"]["lr_d"]
    trainer.betas = tuple(state["hyper"]["betas"])
    trainer.G.dropout_seed, trainer.G.dropout_calls = state["dropout"]["seed"], state["dropout"]["calls"]
    if restore_rng:
        _set_rng_state(state["rng"], trainer.dev)
    if trainer.world > 1:
        trainer.sync_replicas()
    return state.get("extra", {})


def siamese_state(engine, extra: Optional[dict] = None) -> dict:
    torch.cuda.synchronize(engine.dev)
    return {"format": FORMAT, "kind": "siamese", "channels": {"n_channels": engine.n_channels},
            "n_classes": engine.n_classes, "net": _net_state(engine),
            "rng": _rng_state(engine.dev), "extra": extra or {}}


def load_siamese_state(engine, state: dict, restore_rng: bool = True) -> dict:
    if state.get("format") != FORMAT or state.get("kind") != "siamese":
        raise ValueError("not a gap_b200 siamese checkpoint")
    ch = state.get("channels", {"n_channels": 3}).get("n_channels", 3)
    if ch != engine.n_channels:
        raise ValueError(f"checkpoint was written by a Siamese U-Net with n_channels={ch}; this one has "
                         f"n_channels={engine.n_channels}")
    k = state.get("n_classes", 1)           # checkpoints written before multi-class support are n_classes = 1 runs
    if k != engine.n_classes:
        raise ValueError(f"checkpoint was written by a Siamese U-Net with n_classes={k}; this one has "
                         f"n_classes={engine.n_classes}")
    _load_net(engine, state["net"])
    if restore_rng:
        _set_rng_state(state["rng"], engine.dev)
    return state.get("extra", {})


def save(path, state: dict) -> None:
    torch.save(state, path)


def load(path) -> dict:
    return torch.load(path, map_location="cpu", weights_only=False)


def export_reference_state_dicts(state: dict) -> Dict[str, Dict[str, torch.Tensor]]:
    """The reference-format state_dicts inside a checkpoint: {"generator": ..., "discriminator": ...} (what
    train_gan.py:152-153 saves) or {"model": ...} (train.py:311)."""
    if state["kind"] == "pix2pix":
        return {"generator": state["G"]["state_dict"], "discriminator": state["D"]["state_dict"]}
    return {"model": state["net"]["state_dict"]}
