"""C++ host runtime (libodbhost.so): safetensors reader and the prefetching synthetic-token generator."""
import os

import pytest
import torch

from opendiloco_b200 import _lib
from opendiloco_b200.utils import safetensors_io as st
from opendiloco_b200.utils.data import NativeTokenLoader, SyntheticTokenLoader, collate_causal_lm, FakeTokenizedDataset

needs_host = pytest.mark.skipif(_lib.host_lib() is None, reason="libodbhost.so not built")


def test_safetensors_roundtrip(tmp_path):
    t = {"a.weight": torch.randn(7, 5), "b": torch.arange(12, dtype=torch.int64).reshape(3, 4), "c": torch.randn(9).to(torch.bfloat16)}
    p = str(tmp_path / "x.safetensors")
    st.save_safetensors(t, p, metadata={"format": "pt"})
    back = st.load_safetensors(p)
    assert set(back) == set(t) and all(torch.equal(back[k], t[k]) for k in t)
    hf = pytest.importorskip("safetensors.torch")
    ref = hf.load_file(p)                       # the file is a valid safetensors file for the reference's loader too
    assert all(torch.equal(ref[k], t[k]) for k in t)


@needs_host
def test_native_safetensors_matches_python_and_validates(tmp_path, ref_model_dir):
    path = os.path.join(ref_model_dir, "model.safetensors")
    a = st._load_native(path)
    header, base = st.read_header(path)
    assert len(a) == 21 and set(a) == {k for k in header if k != "__metadata__"}
    bad = tmp_path / "bad.safetensors"
    bad.write_bytes(b"\x10\x00\x00\x00\x00\x00\x00\x00" + b'{"x":{"dtype":"F32","shape":[4],"data_offsets":[0,16]}}'[:16])
    with pytest.raises(ValueError):
        st._load_native(str(bad))


@needs_host
def test_native_token_loader_is_deterministic_and_resumable():
    a = NativeTokenLoader(4, 64, 1024, seed=3, rank=1, nbuf=4, pin_memory=False)
    first = [next(a)["input_ids"].clone() for _ in range(6)]
    assert all(int(x.min()) >= 3 and int(x.max()) < 1024 for x in first) and not torch.equal(first[0], first[1])
    sd = a.state_dict()
    nxt = next(a)["input_ids"].clone()
    b = NativeTokenLoader(4, 64, 1024, seed=3, rank=1, nbuf=4, pin_memory=False)
    assert torch.equal(next(b)["input_ids"], first[0])
    b.load_state_dict(sd)
    assert torch.equal(next(b)["input_ids"], nxt)
    c = NativeTokenLoader(4, 64, 1024, seed=3, rank=2, nbuf=4, pin_memory=False)
    assert not torch.equal(next(c)["input_ids"], first[0])          # ranks see different streams
    a.close(), b.close(), c.close()


def test_python_loader_and_collation():
    ld = SyntheticTokenLoader(2, 16, 100, seed=1, pin_memory=False)
    x = next(ld)
    sd = ld.state_dict()
    y = next(ld)["input_ids"].clone()
    ld.load_state_dict(sd)
    assert torch.equal(next(ld)["input_ids"], y) and x["attention_mask"].all()
    it = iter(FakeTokenizedDataset(8, 50, seed=0))
    feats = [next(it), next(it)]
    feats[1] = {"input_ids": feats[1]["input_ids"][:5], "attention_mask": [1] * 5}
    batch = collate_causal_lm(feats, pad_token_id=2)
    assert batch["input_ids"].shape == (2, 8) and (batch["labels"][1, 5:] == -100).all() and (batch["attention_mask"][1, 5:] == 0).all()


def test_training_utils_fingerprint_schedule_and_inf_probe():
    """utils/training.py: debug fingerprint (reference utils.py:70-80), cosine schedule (transformers optimization.py:134-140)
    and the GradScaler inf probe (reference utils.py:124-135)."""
    import math

    import torch

    from opendiloco_b200.utils.training import (cosine_schedule_with_warmup_lambda, found_inf_grad, get_cosine_schedule_with_warmup,
                                                hash_tensor_content)

    a = torch.arange(64 * 64, dtype=torch.float32).view(64, 64) / 7.0
    h = hash_tensor_content(a)
    assert h == hash_tensor_content(a.clone()) and len(h) == 32
    b = a.clone()
    b[40, 40] += 1.0                       # outside the 31 x 31 fingerprint block
    assert hash_tensor_content(b) == h
    b[3, 3] += 1.0
    assert hash_tensor_content(b) != h

    lam = cosine_schedule_with_warmup_lambda(10, 110)
    assert lam(0) == 0.0 and lam(5) == 0.5 and lam(10) == 1.0
    assert abs(lam(60) - 0.5) < 1e-12 and lam(110) == 0.0
    assert abs(lam(210) - 1.0) < 1e-12     # like the HF lambda, the cosine is not clamped past num_training_steps
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=2.0)
    sched = get_cosine_schedule_with_warmup(opt, 10, 110)
    lrs = []
    for _ in range(12):
        opt.step()
        sched.step()
        lrs.append(opt.param_groups[0]["lr"])
    assert abs(lrs[4] - 1.0) < 1e-12 and abs(lrs[9] - 2.0) < 1e-12
    assert abs(lrs[11] - 2.0 * 0.5 * (1 + math.cos(math.pi * 2 / 100))) < 1e-12

    class _Scaler:                          # the two attributes found_inf_grad reads
        def __init__(self, enabled, states):
            self._enabled, self._per_optimizer_states = enabled, states

        def is_enabled(self):
            return self._enabled

    assert found_inf_grad(opt, None) is False
    assert found_inf_grad(opt, _Scaler(False, {})) is False
    assert found_inf_grad(opt, _Scaler(True, {})) is False
    ok = {id(opt): {"found_inf_per_device": {"cpu": torch.tensor(0.0)}}}
    bad = {id(opt): {"found_inf_per_device": {"cpu": torch.tensor(1.0)}}}
    assert found_inf_grad(opt, _Scaler(True, ok)) is False
    assert found_inf_grad(opt, _Scaler(True, bad)) is True


def test_init_weights_writes_a_loadable_hf_checkpoint(tmp_path):
    """init_weights CLI (reference open_diloco/init_weights.py:10-25): config.json + model.safetensors with HF names,
    deterministic in the seed, loadable by this framework and by transformers' LlamaForCausalLM."""
    import json

    import torch

    from opendiloco_b200.init_weights import main as init_main
    from opendiloco_b200.models.llama import LlamaForCausalLM
    from opendiloco_b200.utils.safetensors_io import load_safetensors

    out = tmp_path / "llama-2m-fresh"
    init_main(["--config-name-or-path", "2m", "--save-to-disk", str(out), "--seed", "3"])
    cfg = json.loads((out / "config.json").read_text())
    assert cfg["hidden_size"] == 64 and cfg["num_hidden_layers"] == 2
    sd = load_safetensors(str(out / "model.safetensors"))
    assert "model.embed_tokens.weight" in sd and "lm_head.weight" in sd and "model.layers.1.mlp.down_proj.weight" in sd
    m1 = LlamaForCausalLM.from_pretrained(str(out), device="cpu", precision="32-true")
    m2 = LlamaForCausalLM(m1.config, device="cpu", precision="32-true", seed=3)
    assert torch.equal(m1.arena.master, m2.arena.master)
    transformers = pytest.importorskip("transformers")
    hf = transformers.LlamaForCausalLM.from_pretrained(str(out), torch_dtype=torch.float32)
    ids = torch.randint(0, m1.config.vocab_size, (2, 16))
    with torch.no_grad():
        ref = hf(input_ids=ids, labels=ids).loss
        ours = m1(input_ids=ids, labels=ids).loss
    assert abs(float(ref) - float(ours)) < 1e-4


@needs_host
def test_native_rendezvous_board():
    """csrc/host/rendezvous.cc: key-value records, atomic counters, prefix counts, heartbeats with expiry, the store
    adapter the progress tracker uses - two clients against one in-process server."""
    import threading
    import time

    from opendiloco_b200.parallel import rendezvous as rdv

    assert rdv.available()
    assert rdv.parse_address("odb://127.0.0.1:29400") == ("127.0.0.1", 29400) and rdv.parse_address("/ip4/1.2.3.4") is None
    server = rdv.RendezvousServer(0)
    a = rdv.RendezvousClient("127.0.0.1", server.port, peer_id="worker-0")
    b = rdv.RendezvousClient("127.0.0.1", server.port, peer_id="worker-1")
    try:
        a.set("diloco_progress/worker-0", "3,128,55.5,1.0")
        assert b.get("diloco_progress/worker-0") == b"3,128,55.5,1.0" and b.get("missing") is None
        big = bytes(range(256)) * 64                          # larger than the first receive buffer
        a.set("blob", big)
        assert b.get("blob") == big
        # arrival counter of an outer step, hammered from two threads
        def bump(c):
            for _ in range(200):
                c.add("arrive/7", 1)
        ts = [threading.Thread(target=bump, args=(c,)) for c in (a, b)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert a.add("arrive/7", 0) == 400
        a.set("run/arrive/0/0", "1")
        b.set("run/arrive/0/1", "1")
        assert a.count("run/arrive/0/") == 2 and a.wait(["run/arrive/0/0", "run/arrive/0/1"], 1.0)
        assert not a.wait(["run/arrive/1/0"], 0.05)
        assert b.delete("run/arrive/0/1") and not b.delete("run/arrive/0/1") and a.count("run/arrive/0/") == 1
        # liveness: b beats once with a short ttl and expires, a keeps a background heartbeat
        a.start_heartbeat(ttl=0.6, period=0.1)
        b.heartbeat(ttl=0.15)
        assert sorted(a.alive_peers()) == ["worker-0", "worker-1"]
        time.sleep(0.3)
        assert a.alive_peers() == ["worker-0"]
        # the store adapter drives the progress tracker
        from opendiloco_b200.parallel.diloco import DiloCoProgressTracker

        class _DHT:
            def __init__(self, store, me):
                self._s, self.peer_id, self.num_peers = store, f"worker-{me}", 2

            def store(self):
                return self._s

            def peer_ids(self):
                return ["worker-0", "worker-1"]

        ta = DiloCoProgressTracker(batch_size=4, num_inner_steps=10, dht=_DHT(a.as_store(), 0), publish=True)
        tb = DiloCoProgressTracker(batch_size=4, num_inner_steps=10, dht=_DHT(b.as_store(), 1), publish=True)
        ta.report_local_progress(0, 8)
        tb.report_local_progress(1, 4)
        g = ta.fetch_global_progress()
        assert g.num_peers == 2 and g.epoch == 1
        assert server.num_keys() >= 4
    finally:
        a.close()
        b.close()
        server.stop()


@needs_host
def test_dht_uses_the_native_board_when_given_an_odb_address():
    from opendiloco_b200.parallel import rendezvous as rdv
    from opendiloco_b200.parallel.swarm import DHT

    server = rdv.RendezvousServer(0)
    try:
        dht = DHT(start=True, initial_peers=[f"odb://127.0.0.1:{server.port}"])
        assert dht.board is not None and dht.alive_peers() == ["worker-0"]
        st = dht.store()
        st.set("k", "v")
        assert st.get("k") == b"v" and st.check(["k"]) and not st.check(["k", "nope"]) and st.add("n", 2) == 2
        dht.shutdown()
        assert dht.board is None
        plain = DHT(start=True)
        assert plain.board is None and plain.alive_peers() == ["worker-0"]
    finally:
        server.stop()


def test_cli_flag_grammar_matches_the_reference_launch_lines():
    """utils/config.py: the flag grammar of the reference's README commands (pydantic_config / cyclopts, SURVEY.md §5.6)
    and the strictness of the config models."""
    from opendiloco_b200.train_fsdp import Config
    from opendiloco_b200.utils.config import parse_argv

    argv = ("--per-device-train-batch-size 16 --total_batch_size=2048 --total-steps 88_000 --lr 4e-4 --path-model 1b --fake-data "
            "--no-torch-compile --sharding-strategy _HYBRID_SHARD_ZERO2 --hv.local-steps 500 --hv.galaxy-size 4 --hv.world-rank 1 "
            "--hv.initial-peers tcp://127.0.0.1:29400 --hv.skip-load-from-peers --ckpt.interval 8000 --ckpt.resume true "
            "--max-steps -1").split()
    raw = parse_argv(argv)
    assert raw["per_device_train_batch_size"] == "16" and raw["total_batch_size"] == "2048" and raw["total_steps"] == "88000"
    assert raw["fake_data"] is True and raw["torch_compile"] is False and raw["max_steps"] == "-1"
    assert raw["hv"] == {"local_steps": "500", "galaxy_size": "4", "world_rank": "1", "initial_peers": "tcp://127.0.0.1:29400",
                         "skip_load_from_peers": True}
    assert raw["ckpt"] == {"interval": "8000", "resume": True}
    cfg = Config(**{k: v for k, v in raw.items() if k != "max_steps"})
    assert cfg.total_steps == 88000 and cfg.lr == 4e-4 and cfg.hv.local_steps == 500 and cfg.hv.galaxy_size == 4
    assert cfg.sharding_strategy == "_HYBRID_SHARD_ZERO2" and cfg.torch_compile is False and cfg.ckpt.interval == 8000
    with pytest.raises(Exception):
        Config(**parse_argv(["--path-model", "2m", "--not-a-flag", "1"]))          # unknown flags are errors
    with pytest.raises(ValueError):
        parse_argv(["positional"])
    with pytest.raises(ValueError):
        parse_argv(["--hv", "x", "--hv.local-steps", "2"])                             # scalar / section conflict


@needs_host
def test_token_file_loader_covers_the_corpus_once_per_epoch(tmp_path):
    """csrc/host/tokenfile.cc: shards are cut into seq_len windows; with the seeded shuffle every window is served exactly
    once per epoch, ranks read disjoint samples, the stream is resumable from one integer, raw uint16 files work too."""
    import numpy as np

    from opendiloco_b200.utils.data import TOKEN_SHARD_MAGIC, TokenFileLoader, write_token_shard

    S = 16
    a = torch.arange(0, 40 * S + 5)                     # 40 windows (+ a dropped tail), tokens identify their position
    b = torch.arange(100_000, 100_000 + 24 * S)         # 24 windows, needs 4-byte storage
    write_token_shard(tmp_path / "a.tok", a)
    write_token_shard(tmp_path / "b.tok", b)
    assert (tmp_path / "a.tok").read_bytes()[:8] == TOKEN_SHARD_MAGIC
    assert (tmp_path / "a.tok").stat().st_size == 32 + 2 * a.numel() and (tmp_path / "b.tok").stat().st_size == 32 + 4 * b.numel()
    with pytest.raises(OSError):
        write_token_shard(tmp_path / "bad.tok", torch.tensor([70000]), bytes_per_token=2)

    world, B = 2, 4
    loaders = [TokenFileLoader(str(tmp_path / "*.tok"), B, S, rank=r, world=world, seed=7, pin_memory=False) for r in range(world)]
    assert loaders[0].windows_per_epoch == 64 and loaders[0].batches_per_epoch == 8
    starts = []
    for _ in range(8):                                  # one epoch
        for ld in loaders:
            batch = next(ld)["input_ids"]
            assert batch.shape == (B, S)
            for row in batch:
                assert torch.equal(row, row[0] + torch.arange(S))        # a window is contiguous text
                starts.append(int(row[0]))
    expected = [int(x) for x in a[: 40 * S : S]] + [int(x) for x in b[::S]]
    assert sorted(starts) == sorted(expected)           # every window exactly once, none twice
    assert starts != sorted(starts)                     # and not in file order
    nxt = [next(ld)["input_ids"].clone() for ld in loaders]              # epoch 2 starts: a different permutation
    assert not torch.equal(nxt[0][:, 0], torch.tensor(starts[:B]))
    # resume: same seed + position => same batches
    st = loaders[0].state_dict()
    want = [next(loaders[0])["input_ids"].clone() for _ in range(3)]
    fresh = TokenFileLoader(str(tmp_path / "*.tok"), B, S, rank=0, world=world, seed=7, pin_memory=False)
    fresh.load_state_dict(st)
    assert all(torch.equal(next(fresh)["input_ids"], w) for w in want)
    # sequential order without shuffle; raw header-less uint16 file
    seq = TokenFileLoader([str(tmp_path / "a.tok")], 2, S, shuffle=False, pin_memory=False)
    assert torch.equal(next(seq)["input_ids"][:, 0], torch.tensor([0, S]))
    np.arange(0, 10 * S, dtype=np.uint16).tofile(tmp_path / "raw.bin")
    raw = TokenFileLoader([str(tmp_path / "raw.bin")], 2, S, shuffle=False, pin_memory=False, raw_bytes_per_token=2)
    assert torch.equal(next(raw)["input_ids"][1], S + torch.arange(S))
    with pytest.raises(ValueError):
        TokenFileLoader([str(tmp_path / "raw.bin")], 64, S, pin_memory=False)          # fewer windows than one batch
    for ld in loaders + [fresh, seq, raw]:
        ld.close()
