"""Model parity on CPU: our hand-scheduled engine vs HF LlamaForCausalLM (the model the reference trains)."""
import os

import numpy as np
import pytest
import torch

from opendiloco_b200 import LlamaConfig, LlamaForCausalLM

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _hf():
    tr = pytest.importorskip("transformers")
    return tr


def test_matches_hf_llama_fp32(ref_model_dir):
    tr = _hf()
    torch.manual_seed(0)
    ours = LlamaForCausalLM.from_pretrained(ref_model_dir, precision="32-true")
    hf = tr.LlamaForCausalLM.from_pretrained(ref_model_dir, attn_implementation="sdpa").float()
    ours.train(), hf.train()
    ids = torch.randint(3, 1024, (2, 48))
    o1, o2 = ours(input_ids=ids, labels=ids), hf(input_ids=ids, labels=ids)
    assert abs(o1.loss.item() - o2.loss.item()) < 1e-5
    o1.loss.backward(), o2.loss.backward()
    hfp = dict(hf.named_parameters())
    for n, p in ours.named_parameters():
        assert torch.allclose(p.grad, hfp[n].grad, atol=2e-6, rtol=1e-4), n
    assert list(ours.state_dict().keys()) == list(hf.state_dict().keys())


def test_matches_stored_hf_outputs(ref_model_dir):
    """Loss and a fixed sample of the gradients HF LlamaForCausalLM computed on the reference's 2M checkpoint (fp32, sdpa,
    CPU; tests/golden/llama-2m-fresh/hf_outputs.npz), so the parity check does not depend on transformers being installed."""
    gold = np.load(os.path.join(GOLDEN, "llama-2m-fresh", "hf_outputs.npz"))
    ours = LlamaForCausalLM.from_pretrained(ref_model_dir, precision="32-true")
    ours.train()
    ids = torch.from_numpy(gold["input_ids"])
    loss = ours(input_ids=ids, labels=ids).loss
    assert abs(loss.item() - float(gold["loss"])) < 1e-5
    loss.backward()
    for n, p in ours.named_parameters():
        got = p.grad.reshape(-1)[torch.from_numpy(gold[f"index:{n}"]).long()]
        assert torch.allclose(got, torch.from_numpy(gold[f"grad:{n}"]), atol=2e-6, rtol=1e-4), n


def test_gqa_matches_hf(tmp_path):
    tr = _hf()
    cfg = LlamaConfig(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=8,
                      num_key_value_heads=2, vocab_size=512)
    ours = LlamaForCausalLM(cfg, precision="32-true", seed=3)
    ours.save_pretrained(str(tmp_path))
    hf = tr.LlamaForCausalLM.from_pretrained(str(tmp_path)).float()
    ids = torch.randint(0, 512, (2, 32))
    labels = ids.clone()
    labels[0, :5] = -100
    l1 = ours(input_ids=ids, labels=labels).loss
    l2 = hf(input_ids=ids, labels=labels).loss
    assert abs(l1.item() - l2.item()) < 1e-5


def test_padding_mask_path_matches_hf(tmp_path):
    tr = _hf()
    cfg = LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=1, num_attention_heads=2, vocab_size=256)
    ours = LlamaForCausalLM(cfg, precision="32-true", seed=5)
    ours.save_pretrained(str(tmp_path))
    hf = tr.LlamaForCausalLM.from_pretrained(str(tmp_path)).float()
    ids = torch.randint(3, 256, (2, 16))
    mask = torch.ones_like(ids)
    mask[1, 10:] = 0                      # right padding
    labels = ids.clone()
    labels[mask == 0] = -100
    l1 = ours(input_ids=ids, attention_mask=mask, labels=labels).loss
    l2 = hf(input_ids=ids, attention_mask=mask, labels=labels).loss
    assert abs(l1.item() - l2.item()) < 1e-5
    l1.backward()


def test_native_and_autograd_paths_agree():
    cfg = LlamaConfig(hidden_size=64, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2, vocab_size=1024)
    a = LlamaForCausalLM(cfg, precision="bf16-mixed", seed=7)
    b = LlamaForCausalLM(cfg, precision="bf16-mixed", seed=7)
    ids = torch.randint(3, 1024, (2, 32))
    (a(input_ids=ids, labels=ids).loss * 0.25).backward()
    b.forward_backward(ids, ids, 0.25)
    assert torch.allclose(a.arena.grad, b.arena.grad, atol=1e-6)


def test_bf16_close_to_fp32():
    cfg = LlamaConfig(hidden_size=64, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2, vocab_size=1024)
    a = LlamaForCausalLM(cfg, precision="32-true", seed=7)
    b = LlamaForCausalLM(cfg, precision="bf16-mixed", seed=7)
    ids = torch.randint(3, 1024, (2, 64))
    la, lb = a.forward_backward(ids, ids), b.forward_backward(ids, ids)
    assert abs(la.item() - lb.item()) < 5e-3
    assert ((a.arena.grad - b.arena.grad).norm() / a.arena.grad.norm()).item() < 2e-2


def test_save_load_roundtrip_and_device_api(tmp_path):
    cfg = LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=1, num_attention_heads=2, vocab_size=256)
    a = LlamaForCausalLM(cfg, seed=11)
    a.save_pretrained(str(tmp_path))
    b = LlamaForCausalLM.from_pretrained(str(tmp_path))
    assert torch.equal(a.arena.master, b.arena.master)
    assert b.to("cpu") is b and b.num_parameters() == sum(p.numel() for p in b.parameters())
    sd = a.state_dict()
    c = LlamaForCausalLM(cfg, seed=12)
    c.load_state_dict(sd)
    assert torch.equal(c.arena.shadow, a.arena.shadow)


def test_activation_hooks_reference_style():
    """Forward hooks on modules named *self_attn / lm_head fire with something that has .norm() (reference utils.py:25-67)."""
    from opendiloco_b200.utils.metrics import register_metrics_hooks

    cfg = LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=2, vocab_size=256)
    m = LlamaForCausalLM(cfg, precision="32-true", seed=0)
    log = {}
    handles = register_metrics_hooks(m, ["self_attn", "lm_head"], log, 1)
    ids = torch.randint(0, 256, (1, 16))
    m(input_ids=ids, labels=ids).loss.backward()
    for h in handles:
        h.remove()
    assert set(log) == {"activation/model.layers.0.self_attn", "activation/model.layers.1.self_attn", "activation/lm_head"}
    full = m(input_ids=ids).logits
    assert abs(float(log["activation/lm_head"]) - full.float().norm().item()) / full.float().norm().item() < 1e-4


def test_loss_curve_matches_the_reference_training_loop(tmp_path):
    """The north-star numerics check in miniature (BASELINE.json: "matching the reference's loss curve on the same synthetic
    tokens and seed within 1e-3"): 30 optimizer steps of the reference's statement sequence (train_diloco_torch.py:272-353:
    HF Llama, loss / accum, clip 1.0, torch AdamW(0.1, (0.9, 0.95)), HF cosine schedule, every H steps pseudo-gradient ->
    SGD(0.7, Nesterov 0.9) on the offloaded copy) against DiLoCoTrainer on the same weights and token stream, fp32, CPU."""
    tr = _hf()
    from opendiloco_b200.trainer import DiLoCoTrainer, TrainerConfig
    from opendiloco_b200.utils.data import SyntheticTokenLoader

    cfg = LlamaConfig(hidden_size=64, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2, vocab_size=1024)
    ours = LlamaForCausalLM(cfg, precision="32-true", seed=5)
    ours.save_pretrained(str(tmp_path))
    hf = tr.LlamaForCausalLM.from_pretrained(str(tmp_path), attn_implementation="sdpa").float().train()
    steps, accum, H, lr = 30, 2, 5, 3e-3

    # ---- reference statement sequence
    inner = torch.optim.AdamW(hf.parameters(), lr=lr, weight_decay=0.1, betas=(0.9, 0.95))
    outer = torch.optim.SGD(hf.parameters(), lr=0.7, momentum=0.9, nesterov=True)
    sched = tr.get_cosine_schedule_with_warmup(inner, num_warmup_steps=4, num_training_steps=60)
    off = [p.data.detach().clone() for p in hf.parameters()]
    data = SyntheticTokenLoader(4, 32, vocab_size=1024, seed=11, with_mask=False, pin_memory=False)
    ref_losses = []
    for step in range(1, steps + 1):
        tot = 0.0
        for _ in range(accum):
            ids = next(data)["input_ids"]
            loss = hf(input_ids=ids, labels=ids).loss / accum
            loss.backward()
            tot += float(loss.detach())
        torch.nn.utils.clip_grad_norm_(hf.parameters(), 1.0)
        inner.step()
        sched.step()
        inner.zero_grad()
        if step % H == 0:
            for po, p in zip(off, hf.parameters()):
                p.grad = po - p.data
                p.data = po
            outer.step()
            outer.zero_grad()
            off = [p.data.detach().clone() for p in hf.parameters()]
        ref_losses.append(tot)

    # ---- this framework
    trainer = DiLoCoTrainer(ours, TrainerConfig(lr=lr, grad_accum=accum, local_steps=H, warmup_steps=4, total_steps=60,
                                                 samples_per_step=8))
    data = SyntheticTokenLoader(4, 32, vocab_size=1024, seed=11, with_mask=False, pin_memory=False)
    our_losses = [float(trainer.train_step(data)) for _ in range(steps)]
    assert trainer.optimizer.local_epoch == steps // H
    worst = max(abs(a - b) for a, b in zip(ref_losses, our_losses))
    assert worst < 1e-3, (worst, ref_losses[-3:], our_losses[-3:])          # measured: 7e-7 (fp32 both sides)
    hfp = dict(hf.named_parameters())
    for n, p in ours.named_parameters():
        assert torch.allclose(p.data, hfp[n].data, atol=2e-4), n


def test_full_shard_arena_gathers_and_releases_compute_weights():
    """ZeRO-3 residency of the compute weights (FULL_SHARD): between uses the arena holds only its shard; ``w()`` refuses
    to hand out weights that are not gathered; a gather / release cycle reproduces the replicated forward-backward bit for bit
    (single-process gloo group: the all-gather degenerates to a copy, the residency logic is what is under test)."""
    import os

    import torch.distributed as dist

    from opendiloco_b200.models.config import LlamaConfig
    from opendiloco_b200.models.llama import LlamaForCausalLM

    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29731")
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        cfg = LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=2, vocab_size=256)
        a = LlamaForCausalLM(cfg, device="cpu", precision="bf16-mixed", seed=4)
        b = LlamaForCausalLM(cfg, device="cpu", precision="bf16-mixed", seed=4)
        b.arena.enable_param_sharding(dist.group.WORLD, 0, b.arena.numel)
        assert b.arena.param_sharded and b.arena.shadow is None and b.arena.shadow_shard.numel() == b.arena.numel
        with pytest.raises(RuntimeError, match="sharded"):
            b.arena.w("lm_head.weight")
        ids = torch.randint(3, 256, (2, 32))
        la, lb = a.forward_backward(ids, ids, 1.0), b.forward_backward(ids, ids, 1.0)
        assert b.arena.shadow is None                       # released again after the backward
        assert torch.equal(la, lb) and torch.equal(a.arena.grad, b.arena.grad)
        b.arena.master.mul_(1.5)
        b.arena.sync_shadow()                               # optimizer / checkpoint path: refresh the SHARD from the master slice
        assert torch.equal(b.arena.shadow_shard.float(), b.arena.master.to(torch.bfloat16).float())
    finally:
        if created:
            dist.destroy_process_group()
