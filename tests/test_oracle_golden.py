"""CPU: the oracle restatement vs the golden vectors produced by the REAL reference
(oracle/gen_golden.py).  This is the pin SURVEY 8(c) asks for."""
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import aot_oracle as O
from oracle import weights as OW

VIDEO = ["aott_256", "aott_raw_257", "r50_aotl_small", "r50_deaotl_small", "deaott_small", "swinb_aotl_small",
         "swinb_deaotl_small", "aott_skip2", "deaott_skip3"]


@pytest.fixture(scope="module")
def ops(golden_dir):
    return torch.load(os.path.join(golden_dir, "ops_attention.pt"))


def test_k1_long_term_attention(ops):
    c = ops["k1"]
    W = {"p." + k: v for k, v in c["sd"].items()}
    o = O._lin(O.multihead_attention(c["Q"], c["K"], c["V"], 8), W, "p.projection")
    assert (o - c["out"]).abs().max().item() < 1e-5


def test_k3_self_attention(ops):
    c = ops["k3"]
    W = {"p." + k: v for k, v in c["sd"].items()}
    X = c["X"]
    core = O.multihead_attention(O._lin(X, W, "p.linear_Q"), O._lin(X, W, "p.linear_K"), O._lin(X, W, "p.linear_V"), 8)
    assert (O._lin(core, W, "p.projection") - c["out"]).abs().max().item() < 1e-5


def test_k2_local_attention(ops):
    c = ops["k2"]
    s = O.local_window_scores(c["q"], c["k"], c["sd"]["relative_emb_k.weight"], c["sd"]["relative_emb_k.bias"], 8)
    p = torch.softmax(s, dim=2)
    h, w = c["q"].shape[-2:]
    assert (p.reshape(1, 8, 225, h * w) - c["attn"]).abs().max().item() < 1e-6
    core = O.local_window_aggregate(p, c["v"], 8, c["sd"]["relative_emb_v"])
    o = F.linear(core, c["sd"]["projection.weight"], c["sd"]["projection.bias"])
    assert (o - c["out"]).abs().max().item() < 1e-5


def test_local_attention_two_formulations_agree():
    """unfold form (used by the engine oracle) vs the tap-by-tap form of SURVEY Appendix C."""
    g = torch.Generator().manual_seed(3)
    for (H, d, dv, relv) in ((8, 32, 32, True), (1, 128, 1024, False)):
        h, w = 10, 17
        q = torch.randn(1, H * d, h, w, generator=g)
        k = torch.randn(1, H * d, h, w, generator=g)
        v = torch.randn(1, H * dv, h, w, generator=g)
        rkw = torch.randn(H * 225, d, 1, 1, generator=g) * 0.1
        rkb = torch.randn(H * 225, generator=g) * 0.1
        rv = torch.randn(H, dv, 225, generator=g) * 0.2 if relv else None
        a = O.local_attention(q, k, v, rkw, rkb, rv, H)
        b = O.local_attention_loop(q, k, v, rkw, rkb, rv, H)
        assert (a - b).abs().max().item() < 1e-5


def test_k1p_gated_propagation(ops):
    c = ops["k1p"]
    o, _ = O.gated_propagation({"p." + k: v for k, v in c["sd"].items()}, "p.", c["Q"], c["K"], c["V"], c["U"],
                               c["size_2d"], False)
    assert (o - c["out"]).abs().max().item() < 1e-5


def test_k2p_local_gated_propagation(ops):
    c = ops["k2p"]
    o, _ = O.local_gated_propagation({"p." + k: v for k, v in c["sd"].items()}, "p.", c["q"], c["k"], c["v"],
                                     c["u"], c["size_2d"])
    assert (o - c["out"]).abs().max().item() < 1e-5


def test_sine_position_embedding(ops):
    c = ops["pos"]
    assert (O.pos_emb_sine(c["h"], c["w"]) - c["out"]).abs().max().item() < 1e-6


@pytest.mark.parametrize("name", VIDEO)
def test_video_vs_reference_golden(name, golden_dir):
    """End-to-end: reference engine outputs (stored) vs oracle engine, teacher-forced."""
    g = torch.load(os.path.join(golden_dir, f"video_{name}.pt"))
    sd = OW.build_state_dict(g["model"], seed=g["seed"], flavour=g["flavour"])
    assert OW.checksum(sd) == g["weights_checksum"], "seeded weights are not reproducible on this machine"
    frames, mask = O.synthetic_video(g["frames"], g["H"], g["W"], g["objs"], seed=1234 + g["seed"])
    eng = O.OracleEngine(sd, O.OracleConfig(g["model"]), long_term_mem_gap=g["gap"],
                         short_term_mem_skip=g.get("skip", 1))
    forced = [l.float() for l in g["ref_labels"]]
    with torch.no_grad():
        lo, labels = O.run_video(eng, frames, mask, g["objs"], tuple(g["out_size"]), forced_masks=forced)
    n = g["objs"] + 1
    for a, b in zip(lo, g["ref_logits_lo"]):
        assert (a[:, :n] - b[:, :n]).abs().max().item() < 1e-4
    mism = sum((a.to(torch.uint8) != b).sum().item() for a, b in zip(labels, g["ref_labels"]))
    total = sum(b.numel() for b in g["ref_labels"])
    assert mism <= 1e-4 * total  # fp32 summation-order ties only (SURVEY Appendix E)


@pytest.mark.parametrize("name", ["r50_aotl_480p", "r50_deaotl_480p", "swinb_aotl_592"])
def test_full_geometry_fixture_pin(name, golden_dir):
    """BASELINE-geometry goldens of the REAL reference (tests/golden/full_*.pt): the oracle pin recorded at generation time
    (whole clip, teacher-forced) and, live, the first propagated frame of the oracle against the stored reference logits."""
    from oracle.fixtures import load_full_labels
    g = torch.load(os.path.join(golden_dir, f"full_{name}.pt"))
    assert g["oracle_pin_max_dlogit"] < 1e-4 and g["oracle_pin_label_mismatch"] <= 1e-5 * g["frames"] * g["out_size"][0] * g["out_size"][1]
    labels = load_full_labels(g)
    assert len(labels) == g["frames"] - 1 and tuple(labels[0].shape[-2:]) == tuple(g["out_size"])
    if name != "r50_aotl_480p":
        return                                   # one live frame is enough for the CPU suite's time budget
    sd = OW.build_state_dict(g["model"], seed=g["seed"], flavour=g["flavour"])
    assert OW.checksum(sd) == g["weights_checksum"]
    frames, mask = O.synthetic_video(2, g["H"], g["W"], g["objs"], seed=1234 + g["seed"])
    eng = O.OracleEngine(sd, O.OracleConfig(g["model"]), long_term_mem_gap=g["gap"])
    with torch.no_grad():
        lo, _ = O.run_video(eng, frames, mask, g["objs"], tuple(g["out_size"]), forced_masks=labels[:1])
    assert (lo[0] - g["ref_logits_lo"][1]).abs().max().item() < 1e-4


def _events_inputs(g):
    frames, full = O.synthetic_video(g["frames"], g["H"], g["W"], 14, seed=g["video_seed"])
    first = torch.where(full <= g["first_objs"], full, torch.zeros_like(full))
    return frames, first, {g["event_frame"]: g["new_label"].float()}


@pytest.mark.parametrize("case", ["aott_multi14_events", "deaott_multi14_events"])
def test_multi_engine_and_new_objects_vs_reference_golden(golden_dir, case):
    """AOTInferEngine / DeAOTInferEngine with 14 objects (2 sub-engines, soft_logit_aggregation) where ids 9..14 first
    appear at frame 2 (second reference frame mid-video, evaluator.py:362-402): reference outputs (stored) vs the oracle."""
    g = torch.load(os.path.join(golden_dir, f"events_{case}.pt"))
    sd = OW.build_state_dict(g["model"], seed=g["seed"])
    assert OW.checksum(sd) == g["weights_checksum"]
    frames, first, new = _events_inputs(g)
    eng = O.OracleInferEngine(sd, O.OracleConfig(g["model"]), long_term_mem_gap=g["gap"])
    with torch.no_grad():
        lo, labels = O.run_video_events(eng, frames, first, g["first_objs"], tuple(g["out_size"]), new_objects=new,
                                        forced_masks=[l.float() for l in g["ref_labels"]])
    assert len(eng.aot_engines) == 2
    for a, b, n in zip(lo, g["ref_logits"], g["live_channels"]):
        assert (a[:, :n] - b).abs().max().item() < 1e-4


def test_float64_oracle_close_to_float32():
    """The fp64 truth used to size tolerances must agree with the fp32 restatement."""
    sd = OW.build_state_dict("aott", seed=1)
    frames, mask = O.synthetic_video(2, 65, 81, 2, seed=5)
    outs = []
    for dt in (torch.float32, torch.float64):
        e = O.OracleEngine(sd, O.OracleConfig("aott"), dtype=dt)
        with torch.no_grad():
            e.add_reference_frame(frames[0], mask, [2], 0)
            e.match_propogate_one_frame(frames[1])
            outs.append(e.decode_current_logits((65, 81))[:, :3].double())
    assert (outs[0] - outs[1]).abs().max().item() < 1e-4


def test_state_dict_contract_against_reference(golden_dir):
    """Our parameter trees expose exactly the reference's state_dict keys/shapes (SURVEY App. F), and every config value we
    mirror equals the reference's (both recorded from the reference in tests/golden/reference_contract.json.gz)."""
    from aot_benchmark_b200 import EngineConfig, build_vos_model
    from oracle.fixtures import load_reference_contract
    ref = load_reference_contract(golden_dir)["models"]
    for m in ["aott", "r50_aotl", "deaott", "r50_deaotl", "swinb_aotl", "swinb_deaotl"]:
        mc = EngineConfig("x", m)
        b = {k: list(v.shape) for k, v in build_vos_model(mc.MODEL_VOS, mc).state_dict().items()}
        assert ref[m]["state_dict"] == b, m
        for k, v in mc.__dict__.items():
            if k not in ("EXP_NAME", "MODEL_NAME"):
                assert ref[m]["config"].get(k) == repr(v), (m, k)
