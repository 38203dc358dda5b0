"""CPU tests of the boundary: the library loads, exports every symbol include/seqdiff_b200.h declares,
the host-side mirror keeps the reference's interface, and nothing computes without a GPU."""
import inspect
import os
import re

import pytest
import torch

from helpers import O, ROOT


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "seqdiff_b200.h")).read()
    return sorted(set(re.findall(r"SEQDIFF_API [\w \*]+?(seqdiff_\w+)\(", src)))


def test_library_exports_every_declared_symbol():
    import seqdiff_b200 as sd
    lib = sd.lib()
    syms = _declared_symbols()
    assert len(syms) >= 13
    for s in syms:
        assert hasattr(lib, s), s
    assert sorted(sd._cabi.PROTOTYPES) == syms  # the ctypes table covers the whole header
    assert lib.seqdiff_abi_version() == 1


def test_operator_entry_points_reject_illegal_forms():
    """seqdiff_op_gemm_ex / seqdiff_op_attention_packed reject the forms no kernel implements before anything reaches the device
    (stand-in pointers, never dereferenced)"""
    import ctypes
    import seqdiff_b200 as sd
    lib = sd.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    BF16, FP16, FP32 = 1, 2, 0
    gemm_bad = {
        "split-K with a residual": (BF16, p, None, None, None, 0, 1, 2),
        "split-K into a 16-bit C": (BF16, None, None, None, None, 0, 0, 4),
        "auto split-K into a 16-bit C": (FP16, None, None, None, None, 0, 0, -1),
        "split-K with GELU": (BF16, None, None, None, None, 1, 1, 2),
        "split_k = 0": (BF16, None, None, None, None, 0, 1, 0),
        "LayerNorm residual without resid": (BF16, None, p, p, p, 0, 1, 1),
        "LayerNorm residual without its affine": (BF16, p, p, None, p, 0, 1, 1),
        "LayerNorm residual with split-K": (BF16, p, p, p, p, 0, 1, 3),
        "residual into a 16-bit C": (BF16, p, None, None, None, 0, 0, 1),
        "fp32 mode": (FP32, None, None, None, None, 0, 1, 1),
    }
    for what, (prec, resid, st, g, b, epi, out_f32, split) in gemm_bad.items():
        rc = lib.seqdiff_op_gemm_ex(prec, 256, 768, 768, p, p, p, resid, st, g, b, epi, out_f32, split, p, None)
        assert rc == 1, what  # SEQDIFF_ERR_INVALID
        assert lib.seqdiff_last_error()

    def attn(prec, B, kv_div, q_off=None, k_off=None, q_len=None, Lk_mask=64):
        return lib.seqdiff_op_attention_packed(prec, B, 2, 64, 64, p, 384, p, 384, p, 384, None, 128, p, Lk_mask, q_off, k_off, q_len,
                                               B * 64, B * 64, kv_div, p, None)
    attn_bad = {
        "a pack in fp32 mode": attn(FP32, 4, 1, p, p, p),
        "B % kv_div != 0 (bf16, padded)": attn(BF16, 4, 3),
        "B % kv_div != 0 (fp16, packed)": attn(FP16, 4, 3, p, p, p),
        "B % kv_div != 0 (fp32)": attn(FP32, 4, 3),
        "kv_div = 0": attn(BF16, 4, 0),
        "a pack without k_off": attn(BF16, 4, 1, p, None, p),
        "key-mask pitch below Lk": attn(BF16, 4, 1, p, p, p, Lk_mask=32),
        "padded form with a pack array": attn(BF16, 4, 1, None, p, None),
        "padded form with another mask pitch": attn(FP32, 4, 1, Lk_mask=128),
    }
    for what, rc in attn_bad.items():
        assert rc == 1, what
        assert lib.seqdiff_last_error()


def test_state_dict_schema_is_the_reference_schema():
    import seqdiff_b200 as sd
    for L, rel in ((128, True), (64, True), (64, False)):
        cfg = O.OracleConfig(max_position_embeddings=L, relative_key=rel)
        pos = "relative_key" if rel else "absolute"
        enc = sd.BertConfig(max_position_embeddings=L, intermediate_size=1024, num_hidden_layers=6, position_embedding_type=pos)
        dec = sd.BertConfig(max_position_embeddings=L, intermediate_size=1024, num_hidden_layers=6, position_embedding_type=pos,
                            is_decoder=True, add_cross_attention=True)
        m = sd.ConditionalBertForDiffusionBase(enc, dec, 20)
        want = O.state_dict_schema(cfg)
        got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        assert got == {k: tuple(v) for k, v in want.items()}
        assert len(got) == (242 if rel else 233)  # SURVEY.md section 8b
        # reference init quirk: decoder_normalize.adaLN_modulation[0] is all-zero (model.py:198)
        assert m.decoder_normalize.adaLN_modulation[0].weight.abs().max() == 0
        assert m.ligand_feature_emb.adaLN_modulation[0].weight.abs().max() > 0


def test_signatures_mirror_the_reference():
    import seqdiff_b200 as sd
    f = inspect.signature(sd.ConditionalBertForDiffusionBase.forward)
    assert list(f.parameters)[1:] == ["timestep", "noised_ligand_seq", "ligand_angle", "ligand_attention_masks", "receptor_seq",
                                      "receptor_angle", "receptor_attention_masks", "ligand_pos_ids", "receptor_pos_ids"]
    s = inspect.signature(sd.sample_p_zs_given_zt_discrete)
    assert list(s.parameters)[:8] == ["t", "s", "noised_data", "pred_noise", "noise_schedule", "transition", "diverse", "is_last_step"]
    d = inspect.signature(sd.denoise)
    assert list(d.parameters)[:5] == ["batch", "model", "noise_schedule", "transition", "diverse"]
    p = inspect.signature(sd.PeptideDiff.__init__)
    assert list(p.parameters)[1:7] == ["encoder_config", "decoder_config", "feature_names", "loss_func", "noise_schedule", "timesteps"]
    assert set(sd.sample.CONFIG) >= {"pocket_ext", "timesteps", "max_seq_len", "noise_schedule", "num_heads", "hidden_size",
                                     "num_hidden_layers", "intermediate_size", "position_embedding_type", "batch_size"}


def test_no_cpu_fallback():
    import seqdiff_b200 as sd
    enc = sd.BertConfig(max_position_embeddings=16, intermediate_size=1024, num_hidden_layers=1, position_embedding_type="relative_key")
    dec = sd.BertConfig(max_position_embeddings=16, intermediate_size=1024, num_hidden_layers=1, position_embedding_type="relative_key",
                        is_decoder=True, add_cross_attention=True)
    m = sd.ConditionalBertForDiffusionBase(enc, dec, 20).eval()
    z = torch.zeros
    with pytest.raises(RuntimeError, match="CUDA"):
        m(z(1, 1), z(1, 16, 20), z(1, 16, 8), torch.ones(1, 16), z(1, 16, 20), z(1, 16, 8), torch.ones(1, 16))
    if not torch.cuda.is_available():
        import ctypes
        h = ctypes.c_void_p()
        cfg = m._config_struct()
        rc = sd.lib().seqdiff_model_create(ctypes.byref(cfg), 0, ctypes.byref(h))
        assert rc != 0 and sd.lib().seqdiff_last_error()  # fails loudly, no silent CPU path


def test_error_behaviour_matches_reference():
    import seqdiff_b200 as sd
    sched = sd.PredefinedNoiseScheduleDiscrete("cosine", 50)
    with pytest.raises(AssertionError):  # utils.py:230 exactly-one-of
        sched.get_alpha_bar()
    with pytest.raises(AssertionError):
        sched.get_alpha_bar(t_normalized=torch.zeros(1, 1), t_int=torch.zeros(1, 1))
    with pytest.raises(FileNotFoundError):
        sd.utils._load_blosum.__wrapped__ if hasattr(sd.utils._load_blosum, "__wrapped__") else None
        data, sd.utils._DATA = sd.utils._DATA, "/nonexistent.npz"
        try:
            sd.BlosumTransition(blosum_path="./definitely_missing.pt")
        finally:
            sd.utils._DATA = data
    p = sd.PeptideDiff(sd.BertConfig(max_position_embeddings=16, intermediate_size=1024, num_hidden_layers=1),
                       sd.BertConfig(max_position_embeddings=16, intermediate_size=1024, num_hidden_layers=1), list(sd.AA_VOCAB),
                       torch.nn.CrossEntropyLoss(), "cosine", 50, lr_scheduler="bogus")
    with pytest.raises(ValueError, match="Unknown lr scheduler"):  # model.py:448
        p.configure_optimizers()
    assert p.timesteps == 50 and hasattr(p, "aa_transition_model") and hasattr(p, "discrete_noise_schedule")


def test_sample_dataset_output_format(tmp_path):
    """reference sample.py:231-257: DataFrame columns and pickle round trip (sampler injected: no GPU here)."""
    import pandas as pd
    import seqdiff_b200 as sd

    def fake(batch, model, sched, trans, diverse, **kw):
        n = len(batch["ids"])
        return batch["ids"], ["ACD"] * n, ["ACE"] * n, [2 / 3] * n

    loader = [{"ids": ["1abc_A", "2xyz_B"]}, {"ids": ["3pqr_C"]}]
    out = tmp_path / "sampled.pkl"
    df = sd.sample_dataset(loader, None, noise_schedule=object(), transition=object(), output_path=str(out), denoise_fn=fake)
    assert list(df.columns) == ["structure_ids", "true_sequence", "predict_sequence", "recovery_rate"]
    assert list(df["structure_ids"]) == ["1abc_A", "2xyz_B", "3pqr_C"]
    back = pd.read_pickle(out)
    assert back.equals(df) and len(back) == 3


def test_header_is_plain_c_and_links(tmp_path):
    """include/seqdiff_b200.h is the boundary a non-Python host binds: it must compile as C99 and a C program must link against the
    shared library (no C++ / torch types in the signatures)."""
    import shutil
    import subprocess
    import seqdiff_b200 as sd
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    src = tmp_path / "hc.c"
    src.write_text('#include "seqdiff_b200.h"\nint main(void) { return seqdiff_abi_version() != SEQDIFF_ABI_VERSION; }\n')
    libdir = os.path.dirname(sd._cabi.LIB_PATH)
    exe = tmp_path / "hc"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-L", libdir,
                        "-l:libseqdiff_b200.so", f"-Wl,-rpath,{libdir}", "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert subprocess.run([str(exe)]).returncode == 0


def test_generated_angles_pipeline_host_logic(tmp_path):
    """reference sample_by_generated_angles.py:54-66,197-202,247-278: pad + chunk the structure model's per-complex angles, swap them
    in as `ligand_angles`, same result table (sampler injected: no GPU here)."""
    import pickle

    import numpy as np
    import seqdiff_b200 as sd
    S = sd.sample
    arrays = [np.full((n, 8), float(n), dtype=np.float32) for n in (3, 5, 2)]
    pk = tmp_path / "angles.pkl"
    pk.write_bytes(pickle.dumps(arrays))
    chunks = S.load_generated_angles(str(pk), max_seq_len=6, batch_size=2)
    assert [tuple(c.shape) for c in chunks] == [(2, 6, 8), (1, 6, 8)]
    assert chunks[0][1, 4, 0] == 5 and chunks[0][1, 5, 0] == 0 and chunks[0][0, 3, 0] == 0
    assert torch.equal(S.load_generated_angles(arrays, 6, 2)[1], chunks[1])
    seen = []

    def fake(batch, model, sched, trans, diverse, **kw):
        seen.append(batch["ligand_angles"].clone())
        n = batch["ligand_angles"].shape[0]
        return [f"id{len(seen)}_{i}" for i in range(n)], ["A"] * n, ["C"] * n, [0.0] * n

    loader = [{"ligand_angles": torch.zeros(2, 6, 8), "ligand_seq": torch.zeros(2, 6, 20)}, {"ligand_angles": torch.zeros(1, 6, 8), "ligand_seq": torch.zeros(1, 6, 20)}]
    df = S.sample_dataset(loader, None, noise_schedule=object(), transition=sd.DiscreteUniformTransition(20), denoise_fn=fake, generated_angles=chunks)
    assert len(df) == 3 and torch.equal(seen[0], chunks[0]) and torch.equal(seen[1], chunks[1])
    assert loader[0]["ligand_angles"].abs().sum() == 0  # the caller's batch is not modified
    with pytest.raises(ValueError, match="do not match"):
        S.denoise_with_generated_angles(loader[0], chunks[1], None, None, None, True, denoise_fn=fake)
