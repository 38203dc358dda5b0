"""CPU tests of the design call and of K backbones per pocket in the structure sampler: argument checks in front of every C call, the
C ABI's own argument checks, and the pocket sharding of p_sample_loop_sharded / design_sharded (world-2 gloo, samplers injected: no
GPU here)."""
import ctypes
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_distributed_cpu import _fake_p_sample_loop, _free_port, _make_batch

BAD = [0, -2, 1.5, True, "2", None]


class _NoModel:
    """any use of the model means a C call was reached"""
    def __getattr__(self, name):
        raise AssertionError(f"model.{name} used before the arguments were checked")


class _StructStub:
    """what design reads of a structure model before its first C call"""
    def __init__(self, L=8):
        self.encoder_config = type("Cfg", (), {"max_position_embeddings": L})()
        self.feature_size = 8

    def __getattr__(self, name):
        raise AssertionError(f"structure model.{name} used before the arguments were checked")


def _never(*a, **kw):
    raise AssertionError("sampler called")


@pytest.mark.parametrize("k", BAD)
def test_bad_counts_raise_before_any_c_call(k):
    import seqdiff_b200 as sd
    SM = sd.structure_model
    batch = _make_batch(3)
    for K1, K2 in ((k, 1), (1, k)):
        with pytest.raises(ValueError, match="num_backbones / num_sequences"):
            sd.design.design(_NoModel(), _NoModel(), batch, K1, K2)
        with pytest.raises(ValueError, match="num_backbones / num_sequences"):
            sd.design.design_tensors(_NoModel(), _NoModel(), batch, K1, K2)
        with pytest.raises(ValueError, match="num_backbones / num_sequences"):
            sd.design_dataset([batch], _NoModel(), _NoModel(), K1, K2, design_fn=_never)
        with pytest.raises(ValueError, match="num_backbones / num_sequences"):
            sd.design_sharded(_NoModel(), _NoModel(), batch, K1, K2, design_fn=_never)
    args = (torch.ones(3, 4), torch.zeros(3, 4, 8), torch.zeros(3, 4, 20), torch.ones(3, 4), torch.zeros(3, 4, 8), 3, None)
    with pytest.raises(ValueError, match="num_samples"):
        SM.p_sample_loop(_NoModel(), *args, num_samples=k)
    with pytest.raises(ValueError, match="num_samples"):
        SM.p_sample_loop_tensors(_NoModel(), *args, num_samples=k)
    with pytest.raises(ValueError, match="num_samples"):
        sd.p_sample_loop_sharded(_NoModel(), *args, sample_fn=_never, num_samples=k)


@pytest.mark.parametrize("why", ["ligand too long", "receptor too long", "ligand mask with a hole", "receptor mask with a hole"])
def test_structure_inputs_are_checked_before_any_c_call(why):
    import seqdiff_b200 as sd
    batch = _make_batch(3)
    for k in ("ligand_attn_mask", "receptor_attn_mask"):
        batch[k] = torch.zeros(3, 12)
        batch[k][:, :5] = 1
    side = "ligand_attn_mask" if why.startswith("ligand") else "receptor_attn_mask"
    if "long" in why:
        batch[side][1, :9] = 1  # 9 valid positions, the structure model has 8
        match = "longer than the structure model"
    else:
        batch[side][2, 3] = 0
        match = "prefix of ones"
    with pytest.raises(ValueError, match=match):
        sd.design.design_tensors(_StructStub(8), _NoModel(), batch, 2, 2)


def test_c_abi_rejects_bad_counts_and_flags():
    """seqdiff_struct_sample_multi checks its counts and flags before it touches the handle (a stand-in pointer is never dereferenced)"""
    import seqdiff_b200 as sd
    lib = sd.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    for P, K, Ll, Lr, flags in ((0, 1, 8, 8, 0), (1, 0, 8, 8, 0), (-1, 4, 8, 8, 0), (4, -1, 8, 8, 0), (1 << 16, 1 << 10, 64, 128, 0),
                                (2, 3, 8, 8, 2), (2, 3, 8, 8, -1)):
        rc = lib.seqdiff_struct_sample_multi(p, 1, P, K, Ll, Lr, 5, p, p, p, p, p, p, None, 0, 0, flags, None, p, None)
        assert rc == 1, (P, K, flags)  # SEQDIFF_ERR_INVALID
        assert lib.seqdiff_last_error()
    assert lib.seqdiff_struct_sample_ex(p, 1, 0, 8, 8, 5, p, p, p, p, p, p, None, 0, 0, 0, None, p, None) == 1


def _fake_design(struct_model, seq_model, batch, K1, K2, x_T=None, seq_x_T=None, graph_id0=0, seq_graph_id0=0, **kw):
    """stands in for design(): one entry per (pocket, backbone, sequence) that encodes both graph ids and both start-state rows"""
    P = batch["ligand_seq"].shape[0]
    assert x_T.shape[0] == P * K1 and seq_x_T.shape[0] == P * K1 * K2
    n = P * K1 * K2
    ids = [batch["structure_ids"]["pdb_id"][i // (K1 * K2)] for i in range(n)]
    bb = [(i // K2) % K1 for i in range(n)]
    angles = [f"s{graph_id0 + i // K2}:{float(x_T[i // K2].sum())}" for i in range(n)]
    pred = [f"q{seq_graph_id0 + i}:{float(seq_x_T[i].sum())}" for i in range(n)]
    return ids, bb, angles, ["T"] * n, pred, [float(seq_graph_id0 + i) for i in range(n)]


def _inputs(n, K1, K2, L=4):
    x_T = torch.arange(n * K1).float()[:, None, None].expand(n * K1, L, 8).contiguous()
    seq_x_T = torch.arange(n * K1 * K2).float()[:, None, None].expand(n * K1 * K2, L, 20).contiguous()
    return x_T, seq_x_T


def _worker(rank, world, port, n, K1, K2, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import seqdiff_b200 as sd
    x_T, seq_x_T = _inputs(n, K1, K2)
    seen = {}

    def spy(s, q_, batch, K1_, K2_, **kw):
        seen.update(P=batch["ligand_seq"].shape[0], gid0=kw["graph_id0"], sgid0=kw["seq_graph_id0"], x_T=kw["x_T"].clone(),
                    seq_x_T=kw["seq_x_T"].clone())
        return _fake_design(s, q_, batch, K1_, K2_, **kw)
    out = sd.design_sharded(None, None, _make_batch(n), K1, K2, design_fn=spy, x_T=x_T, seq_x_T=seq_x_T, graph_id0=100, seq_graph_id0=5000)
    # the structure sampler over pockets: rows [lo*K, hi*K) of the start state / noise, per-sample ligand masks, ids from base + lo*K
    loop_seen = []

    def loop_spy(model, lm, x, rs, rm, ra, T, betas, **kw):
        loop_seen.append((rs.shape[0], lm.shape[0], kw["num_samples"]))
        return _fake_p_sample_loop(model, lm, x, rs, rm, ra, T, betas, **kw)
    xs = torch.arange(n * K1).float()[:, None, None].expand(n * K1, 4, 8).contiguous()
    z = torch.arange(3 * n * K1).float().reshape(3, n * K1, 1, 1).expand(3, n * K1, 4, 8).contiguous() * 1e-6
    hist = sd.p_sample_loop_sharded(None, torch.ones(n * K1, 4), xs, torch.zeros(n, 4, 20), torch.ones(n, 4), torch.zeros(n, 4, 8), 3, None,
                                    sample_fn=loop_spy, graph_id0=10, noise_steps=z, num_samples=K1)
    q.put((rank, out, seen, hist, loop_seen))
    dist.barrier()
    dist.destroy_process_group()


def test_sharding_of_pockets_world2():
    n, K1, K2 = 5, 2, 3  # pockets split 3 + 2
    x_T, seq_x_T = _inputs(n, K1, K2)
    want = _fake_design(None, None, _make_batch(n), K1, K2, x_T=x_T, seq_x_T=seq_x_T, graph_id0=100, seq_graph_id0=5000)
    xs = torch.arange(n * K1).float()[:, None, None].expand(n * K1, 4, 8).contiguous()
    z = torch.arange(3 * n * K1).float().reshape(3, n * K1, 1, 1).expand(3, n * K1, 4, 8).contiguous() * 1e-6
    want_hist = _fake_p_sample_loop(None, None, xs, None, None, None, 3, None, graph_id0=10, noise_steps=z)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n, K1, K2, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=120) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, out, seen, hist, loop_seen in res:
        lo, hi = (0, 3) if rank == 0 else (3, 5)
        assert tuple(out) == tuple(want)  # every rank returns the one-GPU result, in (pocket, backbone, sequence) order
        assert seen["P"] == hi - lo and seen["gid0"] == 100 + lo * K1 and seen["sgid0"] == 5000 + lo * K1 * K2
        assert torch.equal(seen["x_T"], x_T[lo * K1:hi * K1]) and torch.equal(seen["seq_x_T"], seq_x_T[lo * K1 * K2:hi * K1 * K2])
        assert loop_seen == [(hi - lo, (hi - lo) * K1, K1)]
        assert torch.equal(hist, want_hist)


def test_design_dataset_frame(tmp_path):
    import pandas as pd

    import seqdiff_b200 as sd
    x_T, seq_x_T = _inputs(2, 2, 2)
    path = tmp_path / "design.pkl"
    df = sd.design_dataset([_make_batch(2)], None, None, 2, 2, output_path=str(path), design_fn=_fake_design, x_T=x_T, seq_x_T=seq_x_T)
    assert list(df.columns) == ["structure_ids", "true_sequence", "predict_sequence", "recovery_rate", "backbone"]
    assert list(df["structure_ids"]) == ["p0"] * 4 + ["p1"] * 4 and list(df["backbone"]) == [0, 0, 1, 1] * 2
    assert pd.read_pickle(path).equals(df)
