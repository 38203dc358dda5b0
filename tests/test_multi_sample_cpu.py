"""CPU tests of K samples per pocket (num_samples): argument checks in front of the C call, the C ABI's own argument checks, and the
pocket sharding of denoise_sharded (world-2 gloo, sampler injected: no GPU here)."""
import ctypes

import pytest
import torch

from test_distributed_cpu import _free_port, _make_batch

BAD = [0, -2, 1.5, True, "2", None]


class _NoModel:
    """any use of the model means a C call was reached"""
    def __getattr__(self, name):
        raise AssertionError(f"model.{name} used before num_samples was checked")


@pytest.mark.parametrize("k", BAD)
def test_bad_num_samples_raise_before_any_c_call(k):
    import seqdiff_b200 as sd
    batch = _make_batch(3)

    def never(*a, **kw):
        raise AssertionError("sampler called")
    with pytest.raises(ValueError, match="num_samples"):
        sd.denoise_tensors(batch, _NoModel(), None, None, True, num_samples=k)
    with pytest.raises(ValueError, match="num_samples"):
        sd.sample.denoise(batch, _NoModel(), None, None, True, num_samples=k)
    with pytest.raises(ValueError, match="num_samples"):
        sd.sample_dataset([batch], _NoModel(), noise_schedule=object(), transition=object(), denoise_fn=never, num_samples=k)
    with pytest.raises(ValueError, match="num_samples"):
        sd.denoise_sharded(batch, _NoModel(), None, None, True, denoise_fn=never, num_samples=k)


def test_sample_dataset_passes_num_samples_through():
    import seqdiff_b200 as sd
    seen = []

    def fake(batch, model, sched, trans, diverse, **kw):
        seen.append(kw.get("num_samples"))
        n = len(batch["ids"]) * kw.get("num_samples", 1)
        return [batch["ids"][i // kw.get("num_samples", 1)] for i in range(n)], ["A"] * n, ["C"] * n, [0.0] * n
    loader = [{"ids": ["1abc_A", "2xyz_B"]}]
    df = sd.sample_dataset(loader, None, noise_schedule=object(), transition=object(), denoise_fn=fake, num_samples=2)
    assert seen == [2] and list(df.columns) == ["structure_ids", "true_sequence", "predict_sequence", "recovery_rate"]
    assert list(df["structure_ids"]) == ["1abc_A", "1abc_A", "2xyz_B", "2xyz_B"]
    sd.sample_dataset(loader, None, noise_schedule=object(), transition=object(), denoise_fn=fake)
    assert seen == [2, None]  # K = 1 calls the sampler exactly as before


def test_c_abi_rejects_bad_pocket_and_sample_counts():
    """seqdiff_sample_multi checks its counts before it touches the handle (so a stand-in pointer is never dereferenced)"""
    import seqdiff_b200 as sd
    lib = sd.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    for P, K, Ll, Lr in ((0, 1, 8, 8), (1, 0, 8, 8), (-1, 4, 8, 8), (4, -1, 8, 8), (1 << 16, 1 << 10, 64, 128), (1 << 20, 1 << 11, 1, 1)):
        rc = lib.seqdiff_sample_multi(p, 1, P, K, Ll, Lr, 5, p, p, p, p, p, p, p, 1, None, 0, 0, 0, p, None)
        assert rc == 1, (P, K)  # SEQDIFF_ERR_INVALID
        assert lib.seqdiff_last_error()


def _fake_denoise(batch, model, noise_schedule, transition, diverse, graph_id0=0, x_T=None, noise_E_steps=None, num_samples=1, **kw):
    """stands in for the CUDA sampler: one entry per (pocket, sample) that encodes the global graph id, the x_T row and the noise slice"""
    P, L = batch["ligand_seq"].shape[:2]
    K = num_samples
    assert x_T.shape[0] == P * K and noise_E_steps.shape[1] == P * K * L
    ids = [f'{batch["structure_ids"]["pdb_id"][i // K]}_{batch["structure_ids"]["ligand_chain"][i // K]}' for i in range(P * K)]
    pred = [f"g{graph_id0 + i}:{int(x_T[i].sum())}:{float(noise_E_steps[:, i * L:(i + 1) * L].sum())}" for i in range(P * K)]
    true = [f"t{int(batch['ligand_seq'][i // K].sum())}" for i in range(P * K)]
    return ids, true, pred, [float(graph_id0 + i) for i in range(P * K)]


def _inputs(n, K, L=4, T=3):
    x_T = torch.arange(n * K).float()[:, None, None].expand(n * K, L, 20).contiguous()
    E = torch.arange(T * n * K * L * 20).float().reshape(T, n * K * L, 20)
    return x_T, E


def _worker(rank, world, port, n, K, q):
    import os

    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import seqdiff_b200 as sd
    x_T, E = _inputs(n, K)
    seen = {}

    def spy(batch, *a, **kw):
        seen.update(P=batch["ligand_seq"].shape[0], gid0=kw["graph_id0"], x_T=kw["x_T"].clone(), E=kw["noise_E_steps"].clone())
        return _fake_denoise(batch, *a, **kw)
    out = sd.denoise_sharded(_make_batch(n), None, None, None, True, denoise_fn=spy, x_T=x_T, noise_E_steps=E, graph_id0=100,
                             num_samples=K)
    q.put((rank, out, seen["P"], seen["gid0"], seen["x_T"], seen["E"]))
    dist.barrier()
    dist.destroy_process_group()


def test_denoise_sharded_shards_pockets_world2():
    import torch.multiprocessing as mp
    n, K, L = 5, 3, 4  # pockets split 3 + 2
    x_T, E = _inputs(n, K)
    want = _fake_denoise(_make_batch(n), None, None, None, True, graph_id0=100, x_T=x_T, noise_E_steps=E, num_samples=K)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n, K, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=120) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, out, P, gid0, xs, Es in res:
        lo, hi = (0, 3) if rank == 0 else (3, 5)
        assert tuple(out) == tuple(want)  # every rank returns the one-GPU result, in (pocket, sample) order
        assert P == hi - lo and gid0 == 100 + lo * K
        assert torch.equal(xs, x_T[lo * K:hi * K]) and torch.equal(Es, E[:, lo * K * L:hi * K * L])
