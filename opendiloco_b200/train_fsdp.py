"""Pre-training entry point with the reference's ``train_fsdp.py`` CLI (SURVEY.md §5.6) on the B200-native engine.

    torchrun --nproc_per_node=2 -m opendiloco_b200.train_fsdp --per-device-train-batch-size 8 --total-batch-size 128 \
        --lr 1e-2 --path-model 2m --fake-data --max-steps 20
    # 8 DiLoCo workers x 1 GPU on one box (reference recipe R/README.md:131-148)
    torchrun --nproc_per_node=8 -m opendiloco_b200.train_fsdp --path-model 150m --precision bf16-mixed \
        --per-device-train-batch-size 32 --total-batch-size 512 --hv.local-steps 500 --hv.galaxy-size 8 --fake-data

Differences from the reference driver that are intentional:
  * workers are ranks of ONE NCCL world (``galaxy_size x gpus_per_worker``); ``--hv.world-rank`` is derived from the
    rank unless workers are launched as separate torchruns that meet on ``--hv.initial-peers tcp://host:port``
    (run_training.sh does that);
  * every GPU of a worker performs the outer step on its own copy / ZeRO shard, so the reference's per-tensor
    rank-0 broadcast after each outer step (train_fsdp.py:410-413) does not exist;
  * ``--sharding-strategy`` is honoured together with ``--hv`` (the reference forces NO_SHARD, train_fsdp.py:192-194),
    which is what BASELINE.json config #4 (1B, 4 workers x 2 GPUs ZeRO-2) needs;
  * ``--torch-compile`` / ``--attn-implementation`` are accepted for CLI compatibility and ignored: the model math is
    hand-written sm_100a kernels, there is no tracing compiler on the hot path.
"""
from __future__ import annotations

import math
import os
import time
from functools import partial
from typing import Any, Literal

import torch
import torch.distributed as dist
from pydantic import model_validator

from .models.llama import LlamaForCausalLM
from .optim.fused import FusedAdamW
from .parallel import comm
from .parallel.compression import get_compression_kwargs
from .parallel.diloco import AllReduceStrategy, DiLoCoOptimizer
from .parallel.swarm import DHT, log_visible_maddrs
from .utils.ckpt import (CKPT_PREFIX, CkptConfig, check_checkpoint_path_access, delete_old_checkpoints,
                         get_diloco_rank_dir_name, get_resume_info, load_checkpoint, save_checkpoint)
from .utils.config import BaseConfig, parse_argv
from .utils.data import TEST_VOCAB_SIZE, TokenFileLoader, data_rank, get_fake_dataloader, get_text_dataloader
from .utils.logger import get_logger, make_metric_logger
from .utils.metrics import register_metrics_hooks
from .utils.training import get_cosine_schedule_with_warmup

TARGET_LAYER_ACTIVATIONS = ["self_attn", "lm_head"]
SHARDING = {"FULL_SHARD", "SHARD_GRAD_OP", "NO_SHARD", "HYBRID_SHARD", "_HYBRID_SHARD_ZERO2"}
logger = get_logger()


def log(message: str) -> None:
    logger.info(f"[rank {os.environ.get('LOCAL_RANK', 0)}] {message}")


class HvConfig(BaseConfig):
    outer_lr: float = 0.7
    local_steps: int = 500
    initial_peers: list[str] | None = None
    host_maddrs: list[str] = ["/ip4/0.0.0.0/tcp/0"]
    announce_maddrs: list[str] | None = None
    matchmaking_time: float | None = None
    averaging_timeout: float | None = None
    hivemind_compression: Literal["fp16", "bf16", "scaled-fp16", "uniform8bit", "quantile8bit", "blockwise8bit"] | None = None
    all_reduce_strategy: AllReduceStrategy = AllReduceStrategy.WAIT_FOR_ALL
    timeout_waiting_for_peers: float | None = None
    skip_load_from_peers: bool = False
    world_rank: int | None = None       # derived from the rank when all workers share one torchrun
    galaxy_size: int
    fail_rank_drop: bool = False
    fused_collective: bool | None = None

    @model_validator(mode="before")
    @classmethod
    def _str_to_list(cls, values: dict[str, Any]) -> dict[str, Any]:
        for name in ("initial_peers", "host_maddrs", "announce_maddrs"):
            if isinstance(values.get(name), str):
                values[name] = [values[name]]
        return values


class Config(BaseConfig):
    path_model: str = "PrimeIntellect/llama-150m-fresh"
    torch_compile: bool = True              # accepted, ignored (see module docstring)
    attn_implementation: str = "sdpa"       # accepted, ignored
    # data
    dataset_name_or_path: str = "allenai/c4"
    seq_length: int = 1024
    c4_tiny: bool = False
    num_workers: int = 4
    # optimisation
    lr: float = 4e-4
    total_batch_size: int = 512
    per_device_train_batch_size: int = 32
    warmup_steps: int = 1000
    total_steps: int = 88_000
    sharding_strategy: str = "NO_SHARD"
    precision: Literal["fp16-mixed", "bf16-mixed", "32-true"] = "bf16-mixed"
    # checkpointing / logging
    project: str = "hivemind_debug"
    metric_logger_type: Literal["wandb", "dummy"] = "wandb"
    log_activations_steps: int | None = None
    ckpt: CkptConfig = CkptConfig()
    # DiLoCo ("hv" kept as the flag namespace of the reference)
    hv: HvConfig | None = None
    fake_data: bool = False
    # attention stays inside the EOS-terminated documents of a packed row (tokens: shards concatenate documents)
    document_mask: bool = False
    max_steps: int | None = None
    seed: int = 0


def _setup_world(config: Config) -> comm.Topology:
    """Bring up the process group for either launch style and carve workers x gpus-per-worker."""
    world_env, rank_env = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0))
    hv = config.hv
    peers = hv.initial_peers if hv is not None else None
    if hv is not None and peers and peers[0].startswith("tcp://"):
        assert hv.world_rank is not None, "--hv.world-rank is required when workers are launched separately"
        comm.init_distributed(init_method=peers[0], rank=hv.world_rank * world_env + rank_env, world_size=hv.galaxy_size * world_env)
        return comm.build_topology(galaxy_size=hv.galaxy_size, gpus_per_worker=world_env)
    comm.init_distributed()
    if hv is None:
        # plain data-parallel baseline: one "worker" spanning every GPU
        return comm.build_topology(galaxy_size=1, gpus_per_worker=dist.get_world_size())
    assert dist.get_world_size() % hv.galaxy_size == 0, "WORLD_SIZE must be a multiple of --hv.galaxy-size"
    return comm.build_topology(galaxy_size=hv.galaxy_size, gpus_per_worker=dist.get_world_size() // hv.galaxy_size)


def get_dataloader(config: Config, topo: comm.Topology, vocab_size: int):
    hv = config.hv
    shard, nshards = data_rank(topo.world_rank if hv else None, topo.galaxy_size if hv else None, topo.gpus_per_worker,
                               topo.rank, topo.local_rank)
    if config.fake_data:
        return get_fake_dataloader(config.seq_length, config.per_device_train_batch_size, min(TEST_VOCAB_SIZE, vocab_size),
                                   num_workers=0, seed=config.seed * 100_003 + shard)
    if config.dataset_name_or_path.startswith("tokens:"):
        # pre-tokenised shards (scripts/tokenize_corpus.py): mmap + native prefetch thread, no tokenizer in the loop
        return TokenFileLoader(config.dataset_name_or_path[len("tokens:"):], config.per_device_train_batch_size, config.seq_length,
                               rank=shard, world=nshards, seed=config.seed)
    return get_text_dataloader(config.dataset_name_or_path, "mistralai/Mistral-7B-v0.1", config.seq_length,
                               config.per_device_train_batch_size, shard, nshards, config.num_workers, pad_to_max=True,
                               c4_tiny=config.c4_tiny)


def train(config: Config) -> None:
    if config.sharding_strategy not in SHARDING:
        raise ValueError(f"Invalid sharding_strategy: {config.sharding_strategy}. Choose one of {sorted(SHARDING)}")
    topo = _setup_world(config)
    hv = config.hv
    rank, local_rank = topo.rank, topo.local_rank
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0))) if torch.cuda.is_available() else torch.device("cpu")
    is_logger_rank = rank == 0

    # batch arithmetic of the reference (train_fsdp.py:186-190): total_batch_size is per WORKER
    assert config.total_batch_size % topo.gpus_per_worker == 0
    batch_size = config.total_batch_size // topo.gpus_per_worker
    assert batch_size % config.per_device_train_batch_size == 0
    grad_accum = batch_size // config.per_device_train_batch_size

    resume_from_ckpt, resume_path = get_resume_info(config.ckpt)
    metric_logger = make_metric_logger(config.metric_logger_type, config.project, config.model_dump(mode="json"),
                                       resume=resume_from_ckpt) if is_logger_rank else None
    if hv is not None:
        log(f"DiLoCo enabled: {topo.galaxy_size} workers x {topo.gpus_per_worker} GPU(s), H={hv.local_steps}")
    if local_rank == 0:
        check_checkpoint_path_access(config.ckpt.path, rank, topo.world_rank if hv else None)

    model = LlamaForCausalLM.from_pretrained(config.path_model, device=device, precision=config.precision, seed=config.seed)
    if dist.get_world_size() > 1:          # everyone starts from rank-0 weights: one flat broadcast
        dist.broadcast(model.arena.master, src=0)
        model.arena.sync_shadow()
    train_dataloader = get_dataloader(config, topo, model.config.vocab_size)
    scaler = torch.amp.GradScaler(device.type, enabled=config.precision == "fp16-mixed")

    shard = config.sharding_strategy != "NO_SHARD"
    inner_factory = partial(FusedAdamW, lr=config.lr, weight_decay=0.1, betas=(0.9, 0.95), dp_group=topo.inner_group, shard=shard,
                            shard_params=config.sharding_strategy in ("FULL_SHARD", "HYBRID_SHARD"))
    scheduler_fn = partial(get_cosine_schedule_with_warmup, num_warmup_steps=config.warmup_steps,
                           num_training_steps=config.total_steps)
    ckpt_rank_dir = get_diloco_rank_dir_name(topo.world_rank) if hv is not None else ""

    dht = None
    if hv is not None:
        dht = DHT(start=True, initial_peers=hv.initial_peers, host_maddrs=hv.host_maddrs, announce_maddrs=hv.announce_maddrs,
                  group=topo.outer_group)
        if local_rank == 0:
            log_visible_maddrs(dht.get_visible_maddrs(), only_p2p=False)
        diloco_args = dict(dht=dht, run_id="llama", batch_size=batch_size, num_inner_steps=hv.local_steps,
                           outer_optimizer=partial(torch.optim.SGD, lr=hv.outer_lr, momentum=0.9, nesterov=True),
                           inner_optimizer=inner_factory, scheduler=None, params=model.parameters(),
                           delay_optimizer_step=False, delay_grad_averaging=False, verbose=True,
                           all_reduce_strategy=hv.all_reduce_strategy, timeout_waiting_for_peers=hv.timeout_waiting_for_peers,
                           fused_collective=hv.fused_collective)
        diloco_args.update(get_compression_kwargs(hv.hivemind_compression))
        if hv.averaging_timeout is not None:
            diloco_args["averaging_timeout"] = hv.averaging_timeout
        if hv.matchmaking_time is not None:
            diloco_args["matchmaking_time"] = hv.matchmaking_time
        optimizer = DiLoCoOptimizer(**diloco_args)
        inner = optimizer.inner_optimizer
    else:
        optimizer = inner = inner_factory(model.parameters())
    scheduler = scheduler_fn(inner)

    start_step, last_loss = 0, None
    if resume_from_ckpt:
        last_loss = load_checkpoint(checkpoint_path=os.path.join(resume_path, ckpt_rank_dir), model=model, optimizer=inner,
                                    scheduler=scheduler, outer_optimizer=optimizer.state_averager.optimizer if hv else None,
                                    scaler=scaler, data_loader=train_dataloader, diloco=optimizer if hv else None,
                                    rank=local_rank)
        start_step = scheduler.last_epoch
        log(f"Resumed from checkpoint at step {start_step} with loss {last_loss}")
    model.train()
    if hv is not None and not hv.skip_load_from_peers and not resume_from_ckpt:
        optimizer.load_state_from_peers()

    current_time = time.time()
    log(f"starting from step {start_step}")
    loss_batch = torch.zeros((), dtype=torch.float32, device=device)
    max_num_peers = 0
    log_activations: dict = {}
    use_native = not scaler.is_enabled()

    for step, batch in enumerate(train_dataloader, start=start_step * grad_accum):
        real_step = (step + 1) // grad_accum
        is_accumulating = bool((step + 1) % grad_accum)
        logging_act = config.log_activations_steps is not None and real_step % config.log_activations_steps == 0
        handles = register_metrics_hooks(model, TARGET_LAYER_ACTIVATIONS, log_activations, grad_accum) if logging_act else []

        ids = batch["input_ids"].to(device, non_blocking=True)
        labels = batch["labels"].to(device, non_blocking=True)
        mask = batch.get("attention_mask")
        if use_native:
            loss = model.forward_backward(ids, labels, 1.0 / grad_accum, mask, document_mask=config.document_mask) / grad_accum
        else:   # fp16: loss scaling goes through autograd + GradScaler exactly like the reference (train_fsdp.py:378-383)
            loss = model(input_ids=ids, attention_mask=mask, labels=labels, document_mask=config.document_mask).loss / grad_accum
            scaler.scale(loss).backward()
        loss_batch += loss.detach()
        for h in handles:
            h.remove()
        if is_accumulating:
            continue

        if scaler.is_enabled():
            inner.unscale_(scaler)        # 1/scale + inf check are folded into the fused norm / AdamW kernels (K11)
        model.clip_grad_norm_(1.0)
        if hv is not None:
            optimizer.step(scaler=scaler if scaler.is_enabled() else None)
        elif scaler.is_enabled():
            optimizer.step_scaled(scaler)
        else:
            optimizer.step()
        scaler.update()
        scheduler.step()
        optimizer.zero_grad()

        if is_logger_rank:
            total_samples = real_step * config.total_batch_size
            effective_step = real_step
            if hv is not None:
                effective_step = real_step * topo.galaxy_size
                total_samples *= topo.galaxy_size
            loss_value = loss_batch.item()
            now = time.time()
            metrics = {"Loss": loss_value, "step": real_step, "lr": inner.param_groups[0]["lr"], "Perplexity": math.exp(min(loss_value, 50)),
                       "effective_step": effective_step, "total_samples": total_samples, "time_taken": now - current_time,
                       "tokens_per_second": config.seq_length * config.total_batch_size / max(now - current_time, 1e-9)}
            if hv is not None:
                num_peers = optimizer.tracker.global_progress.num_peers or 1
                max_num_peers = max(max_num_peers, num_peers)
                metrics["outer_lr"] = optimizer.state_averager.optimizer.param_groups[0]["lr"]
                metrics["num_peers"] = num_peers
                if num_peers < max_num_peers:
                    log(f"Lost a diloco worker, num_peers: {num_peers}, galaxy_size: {topo.galaxy_size}")
                    if hv.fail_rank_drop:
                        raise ValueError(f"Lost a diloco worker, num_peers: {num_peers}, galaxy_size: {topo.galaxy_size}")
            if logging_act:
                metrics.update({k: float(v) for k, v in log_activations.items()})
            current_time = time.time()
            metric_logger.log(metrics)
            if hv is None:
                log(f"step: {real_step}, loss: {loss_value}, lr {inner.param_groups[0]['lr']}")
        log_activations = {}

        if config.ckpt.interval is not None and real_step % config.ckpt.interval == 0:
            log(f"saving at step {real_step}, step {step + 1}")
            ckpt_path = os.path.join(config.ckpt.path, f"{CKPT_PREFIX}_{int(real_step)}", ckpt_rank_dir)
            ctx = optimizer.tracker.pause_updates() if hv is not None else _null()
            with ctx:
                save_checkpoint(checkpoint_path=ckpt_path, model=model, optimizer=inner, scheduler=scheduler,
                                outer_optimizer=optimizer.state_averager.optimizer if hv else None, loss=float(loss_batch.item()),
                                scaler=scaler, data_loader=train_dataloader, save_global_state=local_rank == 0,
                                diloco=optimizer if hv else None, rank=local_rank)
            if dist.get_world_size() > 1:
                comm.barrier()
            if rank == 0 and config.ckpt.topk is not None:
                deleted = delete_old_checkpoints(config.ckpt.path, config.ckpt.topk)
                if deleted:
                    log(f"Deleted old checkpoints: {deleted}")
        loss_batch.zero_()
        if config.max_steps is not None and real_step >= config.max_steps:
            break

    log("Training completed.")
    if is_logger_rank:
        metric_logger.finish()
    if hv is not None:
        optimizer.shutdown()


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def main(argv: list[str] | None = None) -> None:
    config = Config(**parse_argv(argv))
    try:
        train(config)
    finally:
        comm.shutdown_distributed()


if __name__ == "__main__":
    main()
