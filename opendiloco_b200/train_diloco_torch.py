"""Self-contained DiLoCo trainer: every rank is one worker (the reference's ``train_diloco_torch.py``, SURVEY.md §3.4 /
C7), on the B200-native engine.  Works on NCCL (GPUs) and on gloo (CPUs - BASELINE.json config #1).

    torchrun --nproc_per_node=8 -m opendiloco_b200.train_diloco_torch --model-name-or-path 150m --precision bf16-mixed \
        --per-device-train-batch-size 32 --batch-size 512 --local-steps 500 --fake-data

CLI = the reference's cyclopts kwargs (train_diloco_torch.py:142-163) plus ``--fake-data`` / ``--max-steps`` /
``--metric-logger-type`` / ``--seed`` for offline use.  Semantics kept from the reference:
``batch_size`` is PER WORKER; outer step every ``local_steps`` optimizer steps = AVG all-reduce of
(theta_outer - theta_local), SGD(lr=outer_lr, momentum 0.9, nesterov) on theta_outer, theta_local <- theta_outer;
single-file ``model_step_<N>.pt`` checkpoints written by rank 0; optional eval loop.
What changed: theta_outer lives in HBM (no CPU offload), ONE flat collective instead of one per tensor, fused kernels.
"""
from __future__ import annotations

import io
import math
import os
import time
from datetime import datetime
from functools import partial
from typing import Literal

import fsspec
import torch
import torch.distributed as dist

from .models.llama import LlamaForCausalLM
from .optim.fused import FusedAdamW
from .parallel import comm
from .parallel.compression import get_compression
from .parallel.diloco import DiLoCoOptimizer
from .parallel.swarm import DHT
from .utils.config import BaseConfig, parse_argv
from .utils.data import TEST_VOCAB_SIZE, TokenFileLoader, get_fake_dataloader, get_text_dataloader
from .utils.logger import get_logger, make_metric_logger
from .utils.metrics import get_grad_norm, register_metrics_hooks
from .utils.training import get_cosine_schedule_with_warmup

logger = get_logger()


class TorchDilocoConfig(BaseConfig):
    batch_size: int = 512
    per_device_train_batch_size: int = 32
    seq_length: int = 1024
    c4_tiny: bool = False
    checkpoint_interval: int | None = None
    checkpoint_path: str = "outputs"
    warmup_steps: int = 1000
    total_steps: int = 88_000
    precision: Literal["fp16-mixed", "bf16-mixed", "32-true"] = "bf16-mixed"
    project: str = "hivemind_debug"
    model_name_or_path: str = "PrimeIntellect/llama-150m-fresh"
    lr: float = 4e-4
    resume_from_checkpoint: str | None = None
    seed_data: int | None = None
    eval_steps: int | None = None
    log_activations_steps: int | None = None
    local_steps: int = 500
    wandb_group: str | None = None
    resume_only_model: bool = False
    outer_lr: float = 0.7
    # additions for offline / test use
    fake_data: bool = False
    token_shards: str | None = None         # glob of pre-tokenised shards (scripts/tokenize_corpus.py) instead of streaming C4
    eval_token_shards: str | None = None
    # attention stays inside the EOS-terminated documents of a packed row (token shards concatenate documents)
    document_mask: bool = False
    max_steps: int | None = None
    metric_logger_type: Literal["wandb", "dummy"] = "wandb"
    seed: int = 0
    compression: str | None = None
    eval_batches: int = 8


def _ckpt_file(cfg: TorchDilocoConfig, date: str, run_id: str, step: int) -> str:
    return os.path.join(cfg.checkpoint_path, date, os.path.basename(cfg.project.rstrip("/")), run_id, f"model_step_{step}.pt")


def save_checkpoint(path: str, real_step: int, model, optimizer: DiLoCoOptimizer, scheduler, loss: float) -> None:
    """Single-file checkpoint (reference train_diloco_torch.py:59-84) + theta_outer, which the reference loses."""
    data = {"model_state_dict": model.state_dict(), "inner_optimizer_state_dict": optimizer.inner_optimizer.state_dict(),
            "outer_optimizer_state_dict": optimizer.state_averager.optimizer.state_dict(),
            "scheduler_state_dict": scheduler.state_dict(), "loss": loss, "step": real_step,
            "theta_outer": optimizer.state_averager.theta_outer.detach().cpu(), "local_epoch": optimizer.local_epoch,
            "samples_accumulated": optimizer.tracker.local_progress.samples_accumulated}
    buf = io.BytesIO()
    torch.save(data, buf)
    with fsspec.open(path, "wb", auto_mkdir=True) as f:
        f.write(buf.getvalue())
    logger.info(f"Checkpoint saved at step {real_step}")


def load_checkpoint(model, optimizer: DiLoCoOptimizer, scheduler, filename: str, resume_only_model: bool):
    with fsspec.open(filename, "rb") as f:
        ckpt = torch.load(io.BytesIO(f.read()), map_location="cpu", weights_only=False)
    sd = {k.replace("module.", ""): v for k, v in ckpt["model_state_dict"].items()}
    model.load_state_dict(sd)
    sa = optimizer.state_averager
    if resume_only_model:
        sa.theta_outer.copy_(sa.theta_local)
        return 0, ckpt["loss"]
    optimizer.inner_optimizer.load_state_dict(ckpt["inner_optimizer_state_dict"])
    scheduler.load_state_dict(ckpt["scheduler_state_dict"])
    sa.optimizer.load_state_dict(ckpt["outer_optimizer_state_dict"])
    sa.reload_optimizer_state()
    sa.theta_outer.copy_(ckpt["theta_outer"] if ckpt.get("theta_outer") is not None else sa.theta_local)
    sa.local_epoch = int(ckpt.get("local_epoch", 0))
    optimizer.tracker.update_epoch(sa.local_epoch)
    optimizer.tracker.report_local_progress(sa.local_epoch, int(ckpt.get("samples_accumulated", 0)))
    return ckpt["step"], ckpt["loss"]


@torch.no_grad()
def evaluate_model(eval_loader, model, max_batches: int, document_mask: bool = False) -> dict:
    """Mean eval loss / perplexity (reference train_diloco_torch.py:87-110; unlike the reference the eval runs in the
    training precision instead of hard-coded fp16 autocast - SURVEY.md §2.7)."""
    model.eval()
    t0, tot, n = time.time(), 0.0, 0
    for batch in eval_loader:
        dev = model.device
        out = model(input_ids=batch["input_ids"].to(dev), attention_mask=batch.get("attention_mask"), labels=batch["labels"].to(dev),
                    document_mask=document_mask)
        tot += float(out.loss)
        n += 1
        if n >= max_batches:
            break
    model.train()
    logger.info(f"Evaluation time: {time.time() - t0:.2f} seconds")
    loss = tot / max(n, 1)
    return {"eval_loss": loss, "eval_perplexity": math.exp(min(loss, 50))}


def main(cfg: TorchDilocoConfig) -> None:
    comm.init_distributed()
    rank, world = dist.get_rank(), dist.get_world_size()
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    device = torch.device("cuda", local_rank) if torch.cuda.is_available() else torch.device("cpu")
    assert cfg.batch_size % cfg.per_device_train_batch_size == 0
    grad_accum = cfg.batch_size // cfg.per_device_train_batch_size
    date = datetime.now().strftime("%Y-%m-%d")
    metric_logger = None
    if rank == 0:
        kw = {"group": cfg.wandb_group} if (cfg.metric_logger_type == "wandb" and cfg.wandb_group) else {}
        metric_logger = make_metric_logger(cfg.metric_logger_type, cfg.project, cfg.model_dump(mode="json"))
    run_id = os.environ.get("WANDB_RUN_ID", "local")

    model = LlamaForCausalLM.from_pretrained(cfg.model_name_or_path, device=device, precision=cfg.precision, seed=cfg.seed)
    if world > 1:                                   # same init everywhere: one flat broadcast (reference: 111, :253-255)
        dist.broadcast(model.arena.master, src=0)
        model.arena.sync_shadow()
    topo = comm.build_topology(galaxy_size=world, gpus_per_worker=1)
    dht = DHT(start=True, group=topo.outer_group) if world > 1 else None
    optimizer = DiLoCoOptimizer(
        dht=dht, run_id=cfg.project, batch_size=cfg.batch_size, num_inner_steps=cfg.local_steps, params=model.parameters(),
        outer_optimizer=partial(torch.optim.SGD, lr=cfg.outer_lr, momentum=0.9, nesterov=True),
        inner_optimizer=partial(FusedAdamW, lr=cfg.lr, weight_decay=0.1, betas=(0.9, 0.95)),
        grad_compression=get_compression(cfg.compression))
    inner = optimizer.inner_optimizer
    scheduler = get_cosine_schedule_with_warmup(inner, cfg.warmup_steps, cfg.total_steps)
    scaler = torch.amp.GradScaler(device.type, enabled=cfg.precision == "fp16-mixed")

    if cfg.fake_data:
        vocab = min(TEST_VOCAB_SIZE, model.config.vocab_size)
        loader = get_fake_dataloader(cfg.seq_length, cfg.per_device_train_batch_size, vocab, seed=cfg.seed * 100_003 + rank)
        eval_loader = get_fake_dataloader(cfg.seq_length, cfg.per_device_train_batch_size, vocab, seed=999_983) if cfg.eval_steps else None
    elif cfg.token_shards is not None:
        # pre-tokenised shards (scripts/tokenize_corpus.py): mmap + native prefetch thread, no tokenizer in the loop
        loader = TokenFileLoader(cfg.token_shards, cfg.per_device_train_batch_size, cfg.seq_length, rank=rank, world=world,
                                 seed=cfg.seed if cfg.seed_data is None else cfg.seed_data)
        eval_loader = TokenFileLoader(cfg.eval_token_shards or cfg.token_shards, cfg.per_device_train_batch_size, cfg.seq_length,
                                      seed=999_983) if cfg.eval_steps else None
    else:
        loader = get_text_dataloader("allenai/c4", "mistralai/Mistral-7B-v0.1", cfg.seq_length, cfg.per_device_train_batch_size,
                                     rank, world, num_workers=0, pad_to_max=False, c4_tiny=cfg.c4_tiny, seed=cfg.seed_data)
        eval_loader = get_text_dataloader("allenai/c4", "mistralai/Mistral-7B-v0.1", cfg.seq_length, cfg.per_device_train_batch_size,
                                          0, 1, num_workers=0, pad_to_max=False, c4_tiny=cfg.c4_tiny,
                                          split="validation") if cfg.eval_steps else None

    start_step = 0
    if cfg.resume_from_checkpoint is not None:
        start_step, last_loss = load_checkpoint(model, optimizer, scheduler, cfg.resume_from_checkpoint, cfg.resume_only_model)
        logger.info(f"Resumed from checkpoint at step {start_step} with loss {last_loss}")
    model.train()
    logger.info(f"starting from step {start_step}")
    loss_batch = torch.zeros((), dtype=torch.float32, device=device)
    native = not scaler.is_enabled()
    log_activations: dict = {}
    handles: list = []

    for step, batch in enumerate(loader, start=start_step * grad_accum):
        real_step = (step + 1) // grad_accum
        boundary = (step + 1) % grad_accum == 0
        log_act = cfg.log_activations_steps is not None and real_step >= cfg.log_activations_steps and \
            real_step % cfg.log_activations_steps == 0
        if log_act and not handles:
            handles = register_metrics_hooks(model, ["self_attn", "lm_head"], log_activations, grad_accum)
        ids, labels = batch["input_ids"].to(device, non_blocking=True), batch["labels"].to(device, non_blocking=True)
        if native:
            loss = model.forward_backward(ids, labels, 1.0 / grad_accum, batch.get("attention_mask"),
                                          document_mask=cfg.document_mask) / grad_accum
        else:
            loss = model(input_ids=ids, attention_mask=batch.get("attention_mask"), labels=labels,
                         document_mask=cfg.document_mask).loss / grad_accum
            scaler.scale(loss).backward()
        loss_batch += loss.detach()
        if not boundary:
            continue
        for h in handles:
            h.remove()
        handles = []
        if scaler.is_enabled():
            inner.unscale_(scaler)
        model.clip_grad_norm_(1.0)
        norms = get_grad_norm(model) if log_act else None
        optimizer.step(scaler=scaler if scaler.is_enabled() else None)      # inner AdamW; outer step every local_steps
        scaler.update()
        scheduler.step()
        optimizer.zero_grad()
        if optimizer.tracker.local_progress.samples_accumulated == 0 and rank == 0:
            logger.info(f"performed outer step at step {real_step} ({optimizer.last_outer_step_seconds * 1e3:.2f} ms)")

        eval_metrics = {}
        if rank == 0 and cfg.eval_steps is not None and real_step % cfg.eval_steps == 0:
            eval_metrics = evaluate_model(eval_loader, model, cfg.eval_batches, cfg.document_mask)
        if rank == 0:
            lv = float(loss_batch.item())
            m = {"Loss": lv, "step": real_step, "lr": inner.param_groups[0]["lr"], "Perplexity": math.exp(min(lv, 50)),
                 "effective_step": real_step * world, "total_samples": real_step * cfg.batch_size * world, **eval_metrics}
            if norms is not None:
                m.update({k: float(v) for k, v in norms.items()})
            if log_act:
                m.update({k: float(v) for k, v in log_activations.items()})
            metric_logger.log(m)
            logger.info(f"step: {real_step}, loss: {lv}, lr {inner.param_groups[0]['lr']}")
        log_activations = {}
        if rank == 0 and cfg.checkpoint_interval is not None and real_step % cfg.checkpoint_interval == 0:
            save_checkpoint(_ckpt_file(cfg, date, run_id, real_step), real_step, model, optimizer, scheduler, float(loss_batch.item()))
        loss_batch.zero_()
        if cfg.max_steps is not None and real_step >= cfg.max_steps:
            break

    logger.info("Training completed.")
    if rank == 0:
        metric_logger.finish()
    optimizer.shutdown()


def cli(argv: list[str] | None = None) -> None:
    cfg = TorchDilocoConfig(**parse_argv(argv))
    try:
        main(cfg)
    finally:
        comm.shutdown_distributed()


if __name__ == "__main__":
    cli()
