"""CPU suite (-m "not gpu"): the oracle against the reference's golden vectors, the host-side layout
logic, and that the C-ABI library loads and exports every symbol include/quark_b200.h declares."""
import json
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _golden(name):
    z = np.load(os.path.join(GOLD, f"h2_{name}.npz"))
    return z, json.loads(str(z["meta"]))


# ----------------------------------------------------------------------------- oracle vs golden
@pytest.mark.parametrize("name", ["small", "mid"])
def test_oracle_reproduces_reference_golden(name):
    """tests/golden/h2_*.npz hold outputs of the REFERENCE's own modules (oracle/make_golden.py);
    the oracle restatement must reproduce them (float stages to 1e-6, codes exactly)."""
    from oracle import hcodec2, weights
    z, meta = _golden(name)
    cfg = meta["cfg"]
    sd = weights.make_h2_state_dict(cfg, meta["seed_w"])
    wav, feat = weights.synth_inputs(cfg, meta["batch"], meta["n_tokens"], meta["seed_x"])
    emb = hcodec2.encoder_forward(sd, cfg["encoder_config"], wav)
    sem = hcodec2.semantic_encoder_forward(sd, cfg["semantic_encoder_config"], feat)
    ac, sc = hcodec2.codec_encode(sd, cfg, wav, feat)
    rec = hcodec2.codec_decode(sd, cfg, ac, sc)
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
    assert rel(emb, torch.from_numpy(z["emb"])) < 1e-6
    assert rel(sem, torch.from_numpy(z["sem"])) < 1e-6
    assert torch.equal(ac, torch.from_numpy(z["acoustic_codes"])) and torch.equal(sc, torch.from_numpy(z["semantic_codes"]))
    assert rel(rec, torch.from_numpy(z["wav_rec"])) < 1e-6
    assert rec.shape[-1] == meta["n_tokens"] * 3840      # decode(encode(x)) length (SURVEY 8c self-check)


def test_oracle_h1_reproduces_reference_golden():
    """H-Codec-1.0 (BASELINE configs[0]): 1 s 16 kHz clip; golden = outputs of the reference's own Codec."""
    from oracle import hcodec1
    z = np.load(os.path.join(GOLD, "h1_full_1s.npz"))
    meta = json.loads(str(z["meta"]))
    c = hcodec1.H1
    sd = hcodec1.make_state_dict(c, meta["seed_w"])
    g = torch.Generator().manual_seed(meta["seed_x"])
    x = 0.1 * torch.randn(1, 1, 16000, generator=g)
    g2 = torch.Generator().manual_seed(meta["seed_x"] + 1)
    f = torch.randn(1, 768, 50, generator=g2)
    feat = torch.sign(f) * f.abs() ** 0.3
    ac, sc = hcodec1.codec_encode(sd, c, x, feat)
    rec = hcodec1.codec_decode(sd, c, ac, sc)
    assert torch.equal(ac, torch.from_numpy(z["acoustic_codes"])) and torch.equal(sc, torch.from_numpy(z["semantic_codes"]))
    assert float((rec - torch.from_numpy(z["wav_rec"])).abs().max()) < 1e-6 and rec.shape == (1, 16000)
    from unified_audio_b200.codec_h1 import CodecH1
    ref = json.load(open(os.path.join(GOLD, "h1_keys.json")))
    mine = {k: list(v.shape) for k, v in CodecH1({}, {}, {}).state_dict().items()}
    assert mine == {k: v for k, v in ref.items() if not k.startswith("semantic_decoder.")}


def test_oracle_h15_reproduces_reference_golden():
    """H-Codec-1.5 adaptive codec (SURVEY 8f.4): the oracle against the outputs of the reference's own modules at the shipped widths
    (fewer layers: tests/golden/h15_shallow.npz; the 32-layer stacks are pinned by oracle/make_golden_h15.py -> h15_pinning_report.json)"""
    from oracle import hcodec15 as o15
    from oracle.make_golden_h15 import synth
    z = np.load(os.path.join(GOLD, "h15_shallow.npz"))
    meta = json.loads(str(z["meta"]))
    c = o15.h15_shallow()
    sd = o15.make_state_dict(c, meta["seed_w"])
    wav, feat = synth(c, meta["batch"], meta["frames"], meta["seed_x"])
    taps = {}
    ac, sc = o15.codec_encode(sd, c, wav, feat, taps)
    assert torch.equal(taps["align"], torch.from_numpy(z["align"]).float()) and torch.equal(taps["n_groups"], torch.from_numpy(z["n_groups"]))
    assert torch.equal(ac, torch.from_numpy(z["acoustic_codes"])) and torch.equal(sc, torch.from_numpy(z["semantic_codes"]))
    assert int((ac < 0).sum()) > 0, "the fixture must contain padded groups (negative length-packed indices)"
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
    assert rel(taps["sem_agg.out"], torch.from_numpy(z["sem_tok"])) < 1e-5 and rel(taps["ac_agg.out"], torch.from_numpy(z["ac_tok"])) < 1e-5
    rec = o15.codec_decode(sd, c, ac, sc)
    assert rec.shape == tuple(z["wav_rec"].shape) and rel(rec, torch.from_numpy(z["wav_rec"])) < 1e-5
    rep = json.load(open(os.path.join(GOLD, "h15_pinning_report.json")))
    full = [r for r in rep["reports"] if r["name"] == "full"][0]
    assert full["acoustic_codes_equal"] and full["semantic_codes_equal"] and full["rec_rel"] < 2e-5
    from unified_audio_b200.codec_h15 import CodecH15
    assert set(CodecH15().state_dict()) == set(o15.param_specs(o15.H15))


def test_oracle_rvq_self_checks():
    """get_output_from_indices(indices) == returned quantized bit-for-bit; fp64 audit agrees on safe margins;
    explicit-recurrence LSTM == ATen LSTM."""
    from oracle import hcodec2, rvq
    g = torch.Generator().manual_seed(0)
    cb = torch.stack([torch.randn(64, 32, generator=g) * 0.5 * 0.8 ** q for q in range(4)], 0)
    x = torch.randn(200, 32, generator=g)
    idx, quant = rvq.rvq_encode(x, cb)
    assert torch.equal(rvq.rvq_decode(idx, cb), quant)
    tidx, margin = rvq.rvq_margin_audit(x, cb, idx)
    safe = margin > 1e-5
    assert bool((idx[safe] == tidx[safe]).all())
    m = rvq.ResidualVQ(dim=32, codebook_size=64, num_quantizers=4).eval()
    for i, l in enumerate(m.layers):
        l._codebook.embed.copy_(cb[i][None])
    q2, i2, _ = m(x[None])
    assert torch.equal(i2[0], idx) and torch.equal(m.get_output_from_indices(i2)[0], quant)
    # -1 == dropped
    idx2 = idx.clone(); idx2[:, 2] = -1
    assert torch.allclose(rvq.rvq_decode(idx2, cb), cb[0][idx[:, 0]] + cb[1][idx[:, 1]] + cb[3][idx[:, 3]])
    sd = {"r.weight_ih_l0": torch.randn(64, 16, generator=g) * 0.2, "r.weight_hh_l0": torch.randn(64, 16, generator=g) * 0.2,
          "r.bias_ih_l0": torch.randn(64, generator=g) * 0.1, "r.bias_hh_l0": torch.randn(64, generator=g) * 0.1}
    xs = torch.randn(2, 7, 16, generator=g)
    assert torch.allclose(hcodec2.lstm_layer(sd, "r.", xs), hcodec2.lstm_layer_aten(sd, "r.", xs), atol=1e-6)


def test_oracle_edge_cases():
    """ragged / minimum sizes: one token, batch 1; encode length must be a multiple of 3840."""
    from oracle import hcodec2, weights
    cfg = weights.h2_small()
    sd = weights.make_h2_state_dict(cfg, 3)
    wav, feat = weights.synth_inputs(cfg, 1, 1, 5)
    ac, sc = hcodec2.codec_encode(sd, cfg, wav, feat)
    assert ac.shape == (1, cfg["quantizer_config"]["num_quantizers"], 1)
    assert hcodec2.codec_decode(sd, cfg, ac, sc).shape == (1, 3840)


# ----------------------------------------------------------------------------- host logic
@pytest.mark.parametrize("name", ["small", "mid"])
def test_state_dict_layout_matches_reference(name):
    """Codec.state_dict() keys/shapes == the reference's own state_dict (minus the training-only
    semantic_decoder), and == oracle/weights.py's independent restatement."""
    from oracle import weights
    from unified_audio_b200.codec import Codec
    _, meta = _golden(name)
    cfg = meta["cfg"]
    ref = json.load(open(os.path.join(GOLD, f"h2_keys_{name}.json")))
    m = Codec(cfg["encoder_config"], cfg["decoder_config"], cfg["quantizer_config"], cfg["semantic_encoder_config"],
              cfg["semantic_decoder_config"])
    mine = {k: list(v.shape) for k, v in m.state_dict().items()}
    assert mine == {k: v for k, v in ref.items() if not k.startswith("semantic_decoder.")}
    assert {k: tuple(v) for k, v in mine.items()} == {k: tuple(v[0]) for k, v in weights.h2_param_specs(cfg).items()}
    # a reference checkpoint (with semantic_decoder.* keys) loads strictly
    sd = weights.make_h2_state_dict(cfg, 1)
    sd["semantic_decoder.conv1.conv.weight"] = torch.zeros(4, 4, 3)
    m.load_state_dict(sd, strict=True)
    assert torch.equal(m.state_dict()["encoder.out.conv.bias"], sd["encoder.out.conv.bias"])


def test_product_path_refuses_cpu():
    """No CPU / PyTorch fallback: the product path must fail loudly without a CUDA device."""
    from oracle import weights
    from unified_audio_b200.codec import Codec
    cfg = weights.h2_small()
    m = Codec(cfg["encoder_config"], cfg["decoder_config"], cfg["quantizer_config"], cfg["semantic_encoder_config"],
              cfg["semantic_decoder_config"])
    m.load_state_dict(weights.make_h2_state_dict(cfg, 1))
    wav, feat = weights.synth_inputs(cfg, 1, 1, 5)
    with pytest.raises((RuntimeError, AssertionError)):
        m.encode(wav, feat)
    with pytest.raises(RuntimeError):
        m(wav, feat)


def test_product_does_not_import_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "unified_audio_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f"{f} imports the oracle"


def test_precision_policies_cover_every_gemm_group():
    from unified_audio_b200.codec import PRECISION_POLICIES
    groups = {"convnext", "lstm_attn", "mlp", "mlp_dec", "conv", "head", "dft"}
    for name, pol in PRECISION_POLICIES.items():
        assert set(pol) == groups, name
    assert all(PRECISION_POLICIES["accurate"].values())


# ----------------------------------------------------------------------------- C ABI
def test_library_builds_loads_and_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "quark_b200.h")).read()
    declared = set(re.findall(r"\b(qb_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"qb_gemm_desc", "qb_rowmap", "qb_half"}
    from unified_audio_b200 import _lib
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.qb_version() >= 100
    # launches are counted per process: without a CUDA device nothing may have been launched; with one, the suite's GPU tests
    # have launched kernels in this process by now
    if not torch.cuda.is_available():
        assert lib.qb_launch_count() == 0


def test_gemm_desc_struct_layout_matches_header():
    """ctypes mirror of qb_gemm_desc must have the C layout (LP64): 8-byte fields + two int32 pairs."""
    import ctypes as C
    from unified_audio_b200._lib import GemmDesc, RowMap
    assert C.sizeof(RowMap) == 32
    assert GemmDesc.taps.offset == 40 and GemmDesc.stride.offset == 44 and GemmDesc.m_per_batch.offset == 48
    assert GemmDesc.residual.offset == 96 and GemmDesc.act.offset == 128 and GemmDesc.out_f32.offset == 136
    assert GemmDesc.dilation.offset == 136 + 3 * 32 and GemmDesc.act_param.offset == 136 + 3 * 32 + 8
    assert GemmDesc.a_cols.offset == 136 + 3 * 32 + 24 and C.sizeof(GemmDesc) == 136 + 3 * 32 + 32


def test_bench_reference_arm_contract():
    """bench.py --impl reference prints one JSON line with the agreed keys (tiny sample)."""
    import subprocess, sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--seconds", "0.16", "--ref-clips", "1"], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "samples/s" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] == "port"


def test_bicodec_oracle_matches_reference_fixture_and_spec_keys():
    """oracle/bicodec.py reproduces the committed outputs of the reference's BiCodec classes (CPU fp32), and the product's
    state-dict layout is the reference's (tests/golden/bicodec_keys.json, dumped from the reference modules)."""
    import numpy as np
    from oracle import bicodec as ob
    from unified_audio_b200.bicodec import BICODEC_CONFIG, bicodec_spec
    z = np.load(os.path.join(GOLD, "bicodec_small.npz"))
    meta = json.loads(str(z["meta"]))
    cfg = ob.bicodec_small()
    sd = ob.make_state_dict(cfg, meta["seed"])
    wav = ob.detokenize(sd, cfg, torch.from_numpy(z["semantic"]), torch.from_numpy(z["global_tokens"]))
    want = torch.from_numpy(z["wav"])
    assert float((wav - want).abs().max() / want.abs().max()) < 1e-5
    keys = json.load(open(os.path.join(GOLD, "bicodec_keys.json")))
    assert BICODEC_CONFIG == ob.BICODEC_FULL
    spec = {k: list(v) for k, v in bicodec_spec(BICODEC_CONFIG).items()}
    assert spec == keys
    assert {k: list(v[0]) for k, v in ob.param_specs(ob.BICODEC_FULL).items()} == keys


def test_oracle_rvq_matches_reference_in_tree_residual_vq():
    """tests/golden/rvq_intree.npz holds indices / reconstructions of the reference's IN-TREE residual VQ
    (HCodec-2.0/vq/core_vq.py ResidualVectorQuantization, oracle/make_golden_rvq.py); the oracle reproduces them exactly."""
    from oracle import rvq
    z = np.load(os.path.join(GOLD, "rvq_intree.npz"))
    x, cb = torch.from_numpy(z["x"]), torch.from_numpy(z["codebooks"])
    idx, quant = rvq.rvq_encode(x, cb)
    assert torch.equal(idx, torch.from_numpy(z["ref_indices"]))
    assert float((rvq.rvq_decode(idx, cb) - torch.from_numpy(z["ref_dequant"])).abs().max()) < 1e-6


def test_oracle_hubert_front_end_matches_fixture():
    """SSL front end (SURVEY 8f.2, groundwork): oracle/hubert.py reproduces transformers.HubertModel's mean hidden state and
    torchaudio's 48k -> 16k resampler on the committed fixture (oracle/make_golden_hubert.py)."""
    from oracle import hubert as oh
    z = np.load(os.path.join(GOLD, "hubert_small.npz"))
    meta = json.loads(str(z["meta"]))
    c = oh.hubert_small()
    sd = oh.make_state_dict(c, meta["seed"])
    hs = oh.hubert_hidden_states(sd, c, torch.from_numpy(z["wav"]))
    mix = torch.stack(hs, 1).mean(1)
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
    assert rel(mix, torch.from_numpy(z["mix"])) < 1e-5 and rel(hs[-1], torch.from_numpy(z["last"])) < 1e-5
    w48 = torch.from_numpy(z["wav48"])
    assert rel(oh.resample(w48), torch.from_numpy(z["resampled"])) < 1e-6
    assert rel(oh.extract_ssl_features(sd, c, w48), torch.from_numpy(z["feats"])) < 1e-5


def test_oracle_wavlm_and_unise_sr_chain():
    """WavLM-base-plus restatement against the transformers fixture, then the whole UniSE SR chain on the oracles:
    wav -> WavLM mean hidden state -> LLM_SFT.generate -> BiCodec.detokenize -> wav (U/model/model.py:175-193)."""
    from oracle import bicodec as ob
    from oracle import hubert as oh
    from oracle import llama
    z = np.load(os.path.join(GOLD, "wavlm_small.npz"))
    meta = json.loads(str(z["meta"]))
    c = oh.wavlm_small()
    sd = oh.wavlm_make_state_dict(c, meta["seed"])
    mix = torch.stack(oh.wavlm_hidden_states(sd, c, torch.from_numpy(z["wav"])), 1).mean(1)
    assert float((mix - torch.from_numpy(z["mix"])).abs().max() / torch.from_numpy(z["mix"]).abs().max()) < 1e-5
    # chain at reduced widths: 0.32 s of 16 kHz audio -> 16 frames -> 32 global + 16 semantic tokens -> 16 * 320 samples
    wav = 0.1 * torch.randn(2, 16 * 320, generator=torch.Generator().manual_seed(1))
    feats = oh.extract_semantic_features(sd, c, wav)
    assert feats.shape == (2, 16, c["hidden"])
    bc = ob.bicodec_small()
    lm_cfg = llama.lm_small(hidden=128, layers=2, heads=2, gsize=4096, ssize=bc["quantizer"]["codebook_size"], feats=c["hidden"])
    lm_sd = llama.make_lm_state_dict(lm_cfg, 3, 1.0)
    gids, sids = llama.sft_generate(lm_sd, lm_cfg, "se", None, feats, feats.shape[1])
    assert gids.shape == (2, 32) and sids.shape == (2, 16)
    # the small BiCodec has 8 global tokens: take the first 8 of the 32 generated (shipped: 32 of 32)
    out = ob.detokenize(ob.make_state_dict(bc, 4), bc, sids, gids[:, None, :bc["speaker"]["token_num"]])
    assert out.shape == (2, 1, 16 * 320) and bool(torch.isfinite(out).all())


def test_c_abi_reports_errors_without_exceptions(lib):
    """Error behaviour of the boundary: bad arguments return a negative code and leave a message in qb_last_error();
    nothing is launched and no C++ exception crosses the ABI (checked here without a GPU: validation precedes every CUDA call)."""
    import ctypes as C
    from unified_audio_b200._lib import GemmDesc
    assert lib.qb_gemm(None, None) < 0 and b"null desc" in lib.qb_last_error()
    d = GemmDesc()                                     # all-zero descriptor: null operands
    assert lib.qb_gemm(C.byref(d), None) < 0 and b"null operand" in lib.qb_last_error()
    one = C.c_void_p(16)                               # non-null dummy pointers: rejected by shape checks before any use
    d.a_hi, d.w_hi, d.a_ld, d.taps, d.stride = one, one, 48, 1, 1
    assert lib.qb_gemm(C.byref(d), None) < 0 and b"multiple of 64" in lib.qb_last_error()
    rc = lib.qb_lm_decode_layer_tc(one, 33, 512, 8, 2048, one, one, one, one, one, one, one, 64, one, one, one, one, one, one, None)
    assert rc < 0 and b"batch must be 1..32" in lib.qb_last_error()
    rc = lib.qb_lm_head_argmax_tc(one, 4, 512, one, one, 100, one, one, one, 8, one, one, one, one, None)
    assert rc < 0 and b"multiple of 16" in lib.qb_last_error()
    rc = lib.qb_snake_planes(one, 0, one, 1, 8, 96, one, None, 64, 8, 0, None)          # C > ld
    assert rc < 0 and b"snake_planes" in lib.qb_last_error()
    assert lib.qb_version() > 0


def test_oracle_adaptive_alignment_matches_reference_fixture():
    """H-Codec-1.5 groundwork (SURVEY 8f.4): similarity alignment / length packing / de-aggregation restatements against
    alignment matrices produced by the reference's own FlexiCodec static methods (oracle/make_golden_adaptive.py)."""
    from oracle import adaptive as oa
    z = np.load(os.path.join(GOLD, "adaptive_alignment.npz"))
    h = torch.from_numpy(z["h"])
    for thr in (0.6, 0.85):
        a, sim, n = oa.similarity_alignment(h, thr, 8)
        assert torch.equal(a, torch.from_numpy(z[f"align_{thr}"]))
        lens = oa.token_lengths(a)
        assert int(lens.max()) <= 8 and bool((lens.sum(1) == h.shape[1]).all())
        codes = torch.randint(0, 1024, (h.shape[0], 4, a.shape[1]))
        plain, l2 = oa.extract_lengths(oa.inject_lengths(codes, lens.clamp(min=1), 1024), 1024)
        assert torch.equal(plain, codes) and torch.equal(l2, lens.clamp(min=1))
        grouped = torch.randn(h.shape[0], 5, a.shape[1]) * (lens > 0)[:, None]
        assert torch.equal(oa.deaggregate(grouped, a)[:, :, : int(lens[0].sum())][0], oa.deaggregate_by_lengths(grouped, lens)[0])


def test_unise_face_host_logic():
    """unise.Model without a GPU: the checkpoint surface (state_dict holds the LM only, under `dnn.`, like model.py:81-91), the
    shape-only mel against the reference's formula (model.py:53-79 evaluated here with torch.stft on the CPU), the segment count of
    the wrap-pad rule, and the refusal to run off the GPU (no fallback)."""
    import math
    from oracle import bicodec as ob
    from oracle import llama
    from unified_audio_b200.bicodec import BiCodec
    from unified_audio_b200.llm import LLM_SFT
    from unified_audio_b200.ssl import SSLFrontEnd
    from unified_audio_b200.unise import SEG_LEN, BiCodecTokenizer, Model
    c = dict(conv_dim=[64] * 7, conv_kernel=[10, 3, 3, 3, 3, 2, 2], conv_stride=[5, 2, 2, 2, 2, 2, 2], hidden=128, layers=2, heads=2,
             ffn=256, pos_k=16, pos_groups=4, eps=1e-5, num_buckets=32, max_distance=80, kind="wavlm")
    lcfg = llama.lm_small(hidden=128, layers=2, heads=2, gsize=4096, ssize=256, feats=128)
    lm = LLM_SFT(num_tasks=lcfg["num_tasks"], task_map=lcfg["task_map"], feats_dim=lcfg["feats_dim"], llm_base_config=lcfg["llm_base_config"])
    lsd = llama.make_lm_state_dict(lcfg, 3, 2.0)
    lm.load_state_dict(lsd, strict=True)
    model = Model(None, tokenizer=BiCodecTokenizer(BiCodec(ob.bicodec_small())), dnn=lm, semantic_model=SSLFrontEnd(c, in_rate=16000))
    keys = set(model.state_dict().keys())
    assert keys == {"dnn." + k for k in lm.state_dict().keys()}
    ckpt = {"dnn." + k: v + 1.0 if v.is_floating_point() else v for k, v in lsd.items()}
    ckpt["tokenizer.model.whatever"] = torch.zeros(1)            # excluded sub-modules of a Lightning checkpoint are ignored
    model.load_state_dict(ckpt)
    k0 = next(iter(lsd))
    assert torch.equal(model.dnn.state_dict()[k0], lsd[k0] + 1.0)
    x = 0.1 * torch.randn(2, 48000 - 77, generator=torch.Generator().manual_seed(4))
    mel = model.stft_logmel(x)
    assert model.mel_like(x).shape == mel.shape == (2, math.ceil((48000 - 77) / 320), 80) and bool(torch.isfinite(mel).all())
    assert model.mel_frames(SEG_LEN) == 250                       # = the LM's semantic_length for a 5 s segment (llm_sft.py:166)
    assert model.forward(None) is None                            # model.py:93-94
    with pytest.raises(RuntimeError):
        model.enhance("se", None, x[:1])
    with pytest.raises(NotImplementedError):
        model.tokenizer.tokenize(x)


def test_unise_test_step_control_flow_matches_reference_fixture(monkeypatch):
    """tests/golden/unise_glue.npz holds what the REFERENCE'S OWN `Model.test_step` (U/model/model.py:170-286, imported and run
    unmodified by oracle/make_golden_unise.py) hands to its wav writer when its four components are the deterministic stand-ins of
    oracle/unise_stubs.py.  `unise.Model._enhance` with the same stand-ins must produce the same waveforms bit for bit: wrap-pad,
    segmenting, 'se' normalisation, enrollment repetition, the se -> tse -> rtse chain of 'ss', trimming, and the sequence of
    generate() calls.  (CPU: the device kernel behind wrap_segments is replaced by the NumPy expression it implements - its own
    parity is tests/test_ssl_gpu.py::test_tokenizer_glue_and_end_to_end.)"""
    import math
    from oracle import unise_stubs as st
    from oracle.make_golden_unise import digest, make_cases
    from unified_audio_b200 import unise

    def wrap_np(src, seg_len):
        pad = math.ceil(src.shape[-1] / seg_len) * seg_len - src.shape[-1]
        return torch.from_numpy(np.pad(src.numpy(), [(0, 0), (0, pad)], "wrap")).reshape(-1, seg_len)
    monkeypatch.setattr(unise, "wrap_segments", wrap_np)
    z = np.load(os.path.join(GOLD, "unise_glue.npz"))
    model = unise.Model(None, tokenizer=st.Tokenizer(), dnn=st.Dnn(), semantic_model=st.SemanticModel())
    for name, (enroll, src) in make_cases().items():
        mode = name.split("_")[0]
        model.dnn.calls = []
        with torch.no_grad():
            out = model._enhance(mode, enroll, src)
        outs = out if isinstance(out, tuple) else (out,)
        assert model.dnn.calls == json.loads(str(z[f"{name}.calls"])), name
        for i, o in enumerate(outs):
            got, want = digest(o.numpy()), z[f"{name}.est{i}"]
            assert got.shape == want.shape and np.array_equal(got, want), f"{name} output {i} differs from the reference's test_step"
    xm = 0.1 * torch.randn(2, 16000 - 77, generator=torch.Generator().manual_seed(21))
    mel = model.stft_logmel(xm)                                          # vs the reference's own stft_logmel on the same input (model.py:53-79)
    assert mel.shape == z["mel.y"].shape == model.mel_like(xm).shape
    assert float((mel - torch.from_numpy(z["mel.y"])).abs().max()) < 1e-4


def test_oracle_lm_control_flow_matches_reference_fixture():
    """tests/golden/lm_reference.npz holds outputs of the REFERENCE'S OWN `LLM_SFT` (U/model/llm/llm_sft.py, llm.py: unmodified
    `__init__`, conditioning prefix, teacher-forced `forward`, `loss_function`, both decoding loops of `generate`, `sample_logits`;
    only `llm_forward` is bound to this image's transformers - oracle/make_golden_lm_reference.py).  The oracle must reproduce them:
    loss and accuracy of the teacher-forced pass, every greedy token for 'se' / 'tse' / 'rtse', the filtered support of sample_logits."""
    from oracle import llama
    z = np.load(os.path.join(GOLD, "lm_reference.npz"))
    meta = json.loads(str(z["meta"]))
    cfg = meta["cfg"]
    sd = llama.make_lm_state_dict(cfg, meta["seed"], meta["gain"])
    mix, enr = torch.from_numpy(z["mix"]), torch.from_numpy(z["enroll"])
    gids, sids = torch.from_numpy(z["gids"]), torch.from_numpy(z["sids"])
    for task in ("se", "tse", "rtse"):
        e = None if task == "se" else enr
        loss, acc = llama.sft_forward(sd, cfg, task, e, mix, gids, sids)
        assert abs(float(loss) - float(z[f"{task}.loss"])) < 1e-5 * abs(float(z[f"{task}.loss"])) and float(acc) == float(z[f"{task}.acc"])
        gg, ss = llama.sft_generate(sd, cfg, task, e, mix, meta["T"])
        assert np.array_equal(gg.numpy(), z[f"{task}.gen_global"]) and np.array_equal(ss.numpy(), z[f"{task}.gen_semantic"]), task
    lg = torch.from_numpy(z["sample.logits"])
    for top_k, top_p, temp in ((50, 0.95, 0.8), (5, 0.5, 1.0), (20, 1.0, 0.3)):
        probs = llama.sample_filter(lg.clone(), temperature=temp, top_k=top_k, top_p=top_p)
        sup = np.unpackbits(z[f"sample.k{top_k}.p{top_p}.t{temp}.support"], axis=1)[:, :lg.shape[1]].astype(bool)
        assert np.array_equal((probs > 0).numpy(), sup)
        assert np.allclose(probs.max(-1).values.numpy(), z[f"sample.k{top_k}.p{top_p}.t{temp}.probs_max"], rtol=1e-5, atol=1e-7)
    rep = json.load(open(os.path.join(GOLD, "lm_reference_pinning_report.json")))
    assert all(rep[t]["tokens_identical"] for t in ("se", "tse", "rtse", "full_config_tse"))


def test_oracle_tokenizer_chain_matches_reference_fixture():
    """tests/golden/tokenizer_small.npz = outputs of the REFERENCE'S OWN `HCodecTokenizer` (H2/audio_tokenizer.py:47-79: unmodified
    pad_wav / extract_ssl_features / tokenize / detokenize over the reference's `vq.Codec`, transformers' HubertModel and torchaudio's
    Resample - oracle/make_golden_tokenizer.py).  The oracle chain must reproduce them: same padding, features (away from the
    compression's singular point at 0), identical acoustic and semantic codes, the same reconstruction."""
    from oracle import hcodec2
    from oracle import hubert as oh
    from oracle import weights
    z = np.load(os.path.join(GOLD, "tokenizer_small.npz"))
    meta = json.loads(str(z["meta"]))
    c, cfg = meta["hubert"], meta["codec_cfg"]
    sd = weights.make_h2_state_dict(cfg, meta["seed_codec"])
    fsd = oh.make_state_dict(c, meta["seed_ssl"])
    wav = torch.from_numpy(z["wav"])
    hop = 3840
    padded = torch.nn.functional.pad(wav, (0, -(-wav.shape[-1] // hop) * hop - wav.shape[-1]))       # audio_tokenizer.py:63-66
    feats = oh.extract_ssl_features(fsd, c, padded)
    fr = torch.from_numpy(z["feats"])
    big = fr.abs() > 0.2 * fr.abs().max()
    assert feats.shape == fr.shape and float((feats - fr).abs()[big].max() / fr.abs().max()) < 1e-4
    ac, sc = hcodec2.codec_encode(sd, cfg, padded, feats.transpose(1, 2))
    assert np.array_equal(ac.numpy(), z["acoustic"]) and np.array_equal(sc.numpy(), z["semantic"])
    rec = hcodec2.codec_decode(sd, cfg, ac, sc)
    assert rec.shape == z["rec"].shape and float((rec - torch.from_numpy(z["rec"])).abs().max() / np.abs(z["rec"]).max()) < 1e-5


def test_bench_optional_legs_respect_the_wall_clock_budget():
    """bench.run_leg: an optional leg is skipped (and says so) once the invocation has used its wall-clock budget, a failing leg is
    recorded without taking the line down, a finished leg carries its wall time."""
    import sys
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench

    class Ctx:
        budget_s = 1.0

        def __init__(self, over):
            self.over = over

        def over_budget(self):
            return self.over

        def elapsed_s(self):
            return 2.0 if self.over else 0.5
    sec = {}
    bench.run_leg(Ctx(True), sec, "late", lambda: dict(value=1))
    assert "skipped" in sec["late"] and "value" not in sec["late"]
    bench.run_leg(Ctx(False), sec, "ok", lambda: dict(value=3))
    assert sec["ok"]["value"] == 3 and "leg_wall_s" in sec["ok"]

    def boom():
        raise ValueError("x")
    bench.run_leg(Ctx(False), sec, "bad", boom)
    assert "ValueError" in sec["bad"]["error"]


def test_bench_dump_outputs_fits_the_budget_with_a_seeded_sample(tmp_path):
    """bench.dump_outputs: float32 files within the byte budget; small outputs whole and exact (integer codes included), the one that
    does not fit replaced by the same seeded sample of its rows on every call, with the sampled row indices beside it."""
    import sys
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(0)
    arrays = dict(acoustic_codes=torch.randint(0, 1024, (8, 16, 5), generator=g), wav_rec=torch.randn(64, 1000, generator=g))
    budget = 40_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=budget)
    assert sorted(os.listdir(tmp_path / "a")) == ["acoustic_codes.npy", "wav_rec.npy", "wav_rec_rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget
    for f in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    codes = np.load(tmp_path / "a" / "acoustic_codes.npy")
    assert codes.dtype == np.float32 and np.array_equal(codes, arrays["acoustic_codes"].numpy())
    rows = np.load(tmp_path / "a" / "wav_rec_rows.npy")
    wav = np.load(tmp_path / "a" / "wav_rec.npy")
    assert wav.dtype == np.float32 and 1 <= len(rows) < 64 and np.all(np.diff(rows) > 0)
    assert np.array_equal(wav, arrays["wav_rec"].numpy()[rows.astype(np.int64)])
    bench.dump_outputs(str(tmp_path / "a"), arrays)                 # whole this time: the earlier sample's row indices go
    assert sorted(os.listdir(tmp_path / "a")) == ["acoustic_codes.npy", "wav_rec.npy"]
    assert np.array_equal(np.load(tmp_path / "a" / "wav_rec.npy"), arrays["wav_rec"].numpy())
