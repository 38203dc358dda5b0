"""CPU tests of the structure sampler's ragged-packing option: the C entry point's flag check, and `packed` reaching the loop function
through structure_model.sample() and p_sample_loop_sharded (one process, and world-2 gloo with the sampler injected: no GPU here)."""
import ctypes
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_distributed_cpu import _fake_p_sample_loop, _free_port


def test_struct_sample_ex_rejects_unknown_flags():
    """seqdiff_struct_sample_ex checks its flags before it touches the handle (so a stand-in pointer is never dereferenced)"""
    import seqdiff_b200 as sd
    lib = sd.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    for flags in (2, 3, 1 << 30, -1):
        rc = lib.seqdiff_struct_sample_ex(p, 1, 2, 8, 8, 5, p, p, p, p, p, p, None, 0, 0, flags, None, p, None)
        assert rc == 1, flags  # SEQDIFF_ERR_INVALID
        assert b"unknown sampling flag" in lib.seqdiff_last_error()


def _spy(seen):
    def fn(*a, **kw):
        seen.append(kw.get("packed"))
        return _fake_p_sample_loop(*a, **{k: v for k, v in kw.items() if k in ("graph_id0", "noise_steps")})
    return fn


@pytest.mark.parametrize("packed", [None, False, True])
def test_packed_reaches_the_loop_function(packed):
    import seqdiff_b200 as sd
    SM = sd.structure_model
    kw = {} if packed is None else {"packed": packed}
    seen = []
    n = 3
    out = sd.p_sample_loop_sharded(None, torch.ones(n, 4), torch.zeros(n, 4, 8), torch.zeros(n, 4, 20), torch.ones(n, 4), torch.zeros(n, 4, 8), 3,
                                   None, sample_fn=_spy(seen), **kw)
    assert out.shape == (3, n, 4, 8) and seen == [packed]

    class DS:
        timesteps = 3
        alpha_beta_terms = {"betas": SM.cosine_beta_schedule(3)}

        def __len__(self):
            return 2

        def __getitem__(self, i):
            return {"ligand_attn_mask": torch.ones(4), "ligand_angles": torch.zeros(4, 8), "receptor_angles": torch.zeros(4, 8),
                    "receptor_seq": torch.zeros(4, 20), "receptor_attn_mask": torch.ones(4)}

        def sample_noise(self, v):
            return v

    def loop(model, ligand_mask, ligand_angle_noise, total_timesteps, **k):
        seen.append(k.get("packed"))
        return ligand_angle_noise[None].repeat(total_timesteps, 1, 1, 1)

    seen.clear()
    res = SM.sample(None, DS(), loop_fn=loop, **kw)
    assert len(res) == 2 and seen == [packed]


def _worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import seqdiff_b200 as sd
    seen = []
    x = torch.arange(n).float()[:, None, None].expand(n, 4, 8).contiguous()
    out = sd.p_sample_loop_sharded(None, torch.ones(n, 4), x, torch.zeros(n, 4, 20), torch.ones(n, 4), torch.zeros(n, 4, 8), 3, None,
                                   sample_fn=_spy(seen), graph_id0=0, packed=True)
    q.put((rank, out, seen))
    dist.barrier()
    dist.destroy_process_group()


def test_p_sample_loop_sharded_passes_packed_to_every_rank():
    n = 5
    x = torch.arange(n).float()[:, None, None].expand(n, 4, 8).contiguous()
    want = _fake_p_sample_loop(None, None, x, None, None, None, 3, None, graph_id0=0)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=120) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, out, seen in res:
        assert seen == [True] and torch.equal(out, want)
