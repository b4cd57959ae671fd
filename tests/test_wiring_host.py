"""CPU tests of the drop-in wiring around a Tacotron2 model (SURVEY.md section 8b / 8f N2): `genvox_b200.install`
keeps the checkpoint contract, `genvox_b200.wiring.enable_data_parallel` shards the data and exchanges gradients
(world_size 2, gloo).  The model is oracle/standin.py's Tacotron2: the reference model's interface around the CPU oracle
decoder."""
import os
import socket
import tempfile

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import genvox_b200
from oracle import standin, synth


def _model(seed):
    return standin.Tacotron2(synth.DecoderDims(), seed=seed)


def test_install_keeps_state_dict_and_checkpoints_load_both_ways():
    model = _model(3)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    ref_decoder_type = type(model.decoder)
    genvox_b200.install(model, precision="bf16")
    assert type(model.decoder) is genvox_b200.Decoder and model.decoder.precision == "bf16"
    after = model.state_dict()
    assert list(after.keys()) == list(before.keys())                       # same names, same order (checkpoint_manager.py:35-37)
    assert all(torch.equal(after[k], before[k]) for k in before)
    # checkpoint written by the installed model -> a fresh reference model, through the model API (tacotron2.py:574-584)
    opt = model.get_optimizer()
    ckpt = model.get_checkpoint_statedicts(optimizer=opt)
    ckpt["iteration"] = 7                                                   # checkpoint_manager.py adds it
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ckpt.pt")
        torch.save(ckpt, path)
        fresh = _model(99)
        assert isinstance(fresh.decoder, ref_decoder_type)
        fresh.load_checkpoint_statedicts(torch.load(path), save_optimizer_dict=True, optimizer=fresh.get_optimizer())
        assert all(torch.equal(fresh.state_dict()[k], before[k]) for k in before)
        # ... and a reference checkpoint -> an installed model
        torch.save(fresh.get_checkpoint_statedicts(optimizer=None), path)
        other = genvox_b200.install(_model(5))
        other.load_checkpoint_statedicts(torch.load(path), save_optimizer_dict=False, optimizer=None)
        assert all(torch.equal(other.state_dict()[k], before[k]) for k in before)
    # train / eval mode follows the swapped module
    model.eval()
    assert not model.decoder.training
    model.train()
    assert model.decoder.training


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _ToySet(torch.utils.data.Dataset):
    """Stands in for TextMelDataset (models/tts/__init__.py:10-30): item i is recognisable by its token values."""

    def __init__(self, n, n_tok=9, T=6):
        self.n, self.n_tok, self.T = n, n_tok, T

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        g = torch.Generator().manual_seed(100 + i)
        return torch.full((self.n_tok,), i % 60, dtype=torch.int64), torch.randn(80, self.T, generator=g)


def _collate(items):
    tok = torch.stack([t for t, _ in items])
    mel = torch.stack([m for _, m in items])
    B, T = mel.shape[0], mel.shape[2]
    gate = torch.zeros(B, T)
    gate[:, -1] = 1.0
    return {"token_padded": tok, "token_lengths": torch.full((B,), tok.shape[1], dtype=torch.int64), "mel_padded": mel,
            "gate_padded": gate, "mel_lengths": torch.full((B,), T, dtype=torch.int64)}


def _dp_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.set_num_threads(2)
        from genvox_b200 import wiring
        model = _model(1)              # identical init on both ranks; oracle decoder (CPU)
        model.get_train_dataloader = lambda dump_dir, num_loader_workers, batch_size: torch.utils.data.DataLoader(
            _ToySet(12), batch_size=batch_size, shuffle=True, collate_fn=_collate)
        wiring.enable_data_parallel(model, rank, world, group=dist.group.WORLD, seed=4)
        loader = model.get_train_dataloader(dump_dir=None, num_loader_workers=0, batch_size=3)
        model.on_epoch(0)
        seen = []
        criterion, optimizer = model.get_criterion(), model.get_optimizer()
        model.train()
        for batch in loader:
            seen += batch["token_padded"][:, 0].tolist()
            model.train_step(batch=batch, criterion=criterion, optimizer=optimizer)      # the reference Trainer's call (:207)
            break
        digest = torch.cat([p.detach().flatten()[:64] for p in model.parameters()])
        out[rank] = (sorted(set(seen)), digest, {k: float(v) for k, v in model.loss_items.items()}, float(model.grad_norm_val))
    finally:
        dist.destroy_process_group()


def test_data_parallel_wiring_world_size_2_gloo():
    world, port = 2, _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_dp_worker, args=(world, port, out), nprocs=world, join=True)
    (seen0, p0, loss0, gn0), (seen1, p1, loss1, gn1) = out[0], out[1]
    assert seen0 and seen1 and not set(seen0) & set(seen1)            # DistributedSampler: disjoint shards
    assert torch.equal(p0, p1)                                        # same averaged gradient -> same parameters after Adam
    assert abs(gn0 - gn1) < 1e-6 * max(gn0, 1.0)                      # clip_grad_norm_ saw the exchanged gradients on both ranks
    assert loss0 != loss1                                             # ... of different local batches
