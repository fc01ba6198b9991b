"""Generate the golden fixtures under tests/golden/ by running the REAL reference.

TEST INFRASTRUCTURE ONLY.  Run in the build container (needs /root/reference, which does not
exist on the GPU box):

    python oracle/gen_golden.py [--out tests/golden] [--only NAME]

For every case it (1) builds a seeded weight set with oracle/weights.py, (2) loads it with
``load_state_dict(strict=True)`` into the reference's own model (this also checks the
state_dict key contract of SURVEY 8b), (3) drives the reference's own eval engine
(``build_engine(..., phase='eval')``) through the evaluator's per-frame protocol
(evaluator.py:315-422) on seeded synthetic clips, (4) stores the reference outputs, and
(5) prints how far oracle/aot_oracle.py is from them (the pin).

The only patch applied to the reference is the one SURVEY 0.4 documents:
``transformer.MultiheadLocalAttentionV3 := attention.MultiheadLocalAttentionV2`` (the
reference's no-sampler fallback V3 is broken at this commit; V2's unfold branch is the
mathematical definition).  Nothing from the reference is copied into the repo.
"""
from __future__ import annotations

import argparse
import os
import sys

import torch
import torch.nn.functional as F

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("AOT_REFERENCE", "/root/reference")
sys.path.insert(0, REPO)
sys.path.insert(0, REF)

from oracle import aot_oracle as O  # noqa: E402
from oracle import weights as OW  # noqa: E402

import networks.layers.attention as RA  # noqa: E402  (reference)
import networks.layers.transformer as RT  # noqa: E402

RT.MultiheadLocalAttentionV3 = RA.MultiheadLocalAttentionV2  # SURVEY 0.4

from configs.default import DefaultEngineConfig  # noqa: E402
from networks.engines import build_engine as ref_build_engine  # noqa: E402
from networks.models import build_vos_model as ref_build_model  # noqa: E402

# name: (model, H, W, out_h, out_w, frames, objs, gap, weight flavour)
VIDEO_CASES = {
    "aott_256": ("aott", 256, 256, 256, 256, 3, 1, 9999, "calibrated"),          # BASELINE configs[0]
    "aott_raw_257": ("aott", 257, 257, 240, 250, 4, 3, 2, "raw"),
    "r50_aotl_small": ("r50_aotl", 161, 241, 150, 230, 7, 10, 2, "calibrated"),
    "r50_deaotl_small": ("r50_deaotl", 161, 241, 150, 230, 7, 10, 2, "calibrated"),
    "deaott_small": ("deaott", 129, 177, 129, 177, 5, 4, 2, "calibrated"),
    # Swin-B encoder (BASELINE configs[3]); align_corners=False models take multiples of 16 (video_transforms.py:649-655).
    # 144x208 -> 36x52 / 18x26 / 9x13 maps: window padding and shifted-window masks at every stage
    "swinb_aotl_small": ("swinb_aotl", 144, 208, 130, 200, 5, 6, 2, "calibrated"),
    "swinb_deaotl_small": ("swinb_deaotl", 112, 176, 112, 176, 4, 3, 2, "calibrated"),
    # TEST_SHORT_TERM_MEM_SKIP = 2: the short-term memory is the frame BEFORE the previous one (aot_engine.py:329-332)
    "aott_skip2": ("aott", 129, 177, 129, 177, 6, 3, 2, "calibrated", 2),
    "deaott_skip3": ("deaott", 113, 145, 113, 145, 6, 2, 3, "calibrated", 3),
}


def run_reference_video(model_name, H, W, oh, ow, T, objs, gap, flavour, skip=1, seed=0):
    torch.manual_seed(0)
    sd = OW.build_state_dict(model_name, seed=seed, flavour=flavour)
    rcfg = DefaultEngineConfig("golden", model_name)
    ref_model = ref_build_model(rcfg.MODEL_VOS, rcfg).eval()
    ref_model.load_state_dict(sd, strict=True)
    engine = ref_build_engine(rcfg.MODEL_ENGINE, phase="eval", aot_model=ref_model, gpu_id=-1,
                              long_term_mem_gap=gap, short_term_mem_skip=skip)
    engine.eval()
    frames, mask = O.synthetic_video(T, H, W, objs, seed=1234 + seed)
    with torch.no_grad():
        logits_lo, labels = O.run_video(engine, frames, mask, objs, (oh, ow))
    return sd, frames, mask, logits_lo, labels


def video_case(name, out_dir):
    model_name, H, W, oh, ow, T, objs, gap, flavour = VIDEO_CASES[name][:9]
    skip = VIDEO_CASES[name][9] if len(VIDEO_CASES[name]) > 9 else 1
    sd, frames, mask, ref_lo, ref_labels = run_reference_video(model_name, H, W, oh, ow, T, objs, gap, flavour, skip)
    # pin the oracle (teacher-forced with the reference's own labels)
    ocfg = O.OracleConfig(model_name)
    oe = O.OracleEngine(sd, ocfg, long_term_mem_gap=gap, short_term_mem_skip=skip)
    with torch.no_grad():
        o_lo, o_labels = O.run_video(oe, frames, mask, objs, (oh, ow), forced_masks=ref_labels)
    max_d = max((a - b).abs().max().item() for a, b in zip(ref_lo, o_lo))
    mism = sum((a != b).sum().item() for a, b in zip(ref_labels, o_labels))
    used = sorted(set(int(v) for l in ref_labels for v in l.unique().tolist()))
    print(f"[{name}] oracle vs reference: max|dlogit|={max_d:.3e} label mismatches={mism} "
          f"|logit|max={max(a[:, :objs + 1].abs().max().item() for a in ref_lo):.2f} labels used={used}")
    torch.save({
        "model": model_name, "H": H, "W": W, "out_size": (oh, ow), "frames": T, "objs": objs, "gap": gap,
        "flavour": flavour, "seed": 0, "skip": skip, "weights_checksum": OW.checksum(sd),
        "ref_logits_lo": [t.to(torch.float32) for t in ref_lo],
        "ref_labels": [t.to(torch.uint8) for t in ref_labels],
        "oracle_pin_max_dlogit": max_d, "oracle_pin_label_mismatch": mism,
    }, os.path.join(out_dir, f"video_{name}.pt"))


# BASELINE geometries (configs[1], [2], [3]) through the REAL reference: name -> (model, H, W, out_h, out_w, frames, objs, gap,
# flavour, propagated frames whose low-res logits are stored).  Labels of every frame are stored zlib-compressed; logits only
# for the listed frames (1.1-1.7 MB each): the first propagated frame, the frame before / at / after the first bank growth.
FULL_CASES = {
    "r50_aotl_480p": ("r50_aotl", 481, 849, 480, 854, 8, 10, 5, "calibrated", (1, 5, 6, 7)),
    "r50_deaotl_480p": ("r50_deaotl", 481, 849, 480, 854, 8, 10, 5, "calibrated", (1, 5, 6, 7)),
    "swinb_aotl_592": ("swinb_aotl", 592, 1040, 592, 1040, 4, 10, 2, "calibrated", (1, 2, 3)),
}


def full_case(name, out_dir):
    import time
    import zlib
    model_name, H, W, oh, ow, T, objs, gap, flavour, keep = FULL_CASES[name]
    t0 = time.time()
    sd, frames, mask, ref_lo, ref_labels = run_reference_video(model_name, H, W, oh, ow, T, objs, gap, flavour)
    t_ref = time.time() - t0
    oe = O.OracleEngine(sd, O.OracleConfig(model_name), long_term_mem_gap=gap)
    with torch.no_grad():
        o_lo, o_labels = O.run_video(oe, frames, mask, objs, (oh, ow), forced_masks=ref_labels)
    max_d = max((a - b).abs().max().item() for a, b in zip(ref_lo, o_lo))
    mism = sum((a != b).sum().item() for a, b in zip(ref_labels, o_labels))
    used = sorted(set(int(v) for l in ref_labels for v in l.unique().tolist()))
    print(f"[{name}] reference ran {T - 1} propagated frames in {t_ref:.1f} s; oracle vs reference: max|dlogit|={max_d:.3e} "
          f"label mismatches={mism} labels used={used}")
    lab = torch.stack([t.to(torch.uint8).reshape(oh, ow) for t in ref_labels]).contiguous()
    torch.save({
        "model": model_name, "H": H, "W": W, "out_size": (oh, ow), "frames": T, "objs": objs, "gap": gap,
        "flavour": flavour, "seed": 0, "weights_checksum": OW.checksum(sd),
        "logit_frames": list(keep), "ref_logits_lo": {int(t): ref_lo[t - 1].to(torch.float32).clone() for t in keep},
        "ref_labels_zlib": zlib.compress(lab.numpy().tobytes(), 9), "ref_labels_shape": tuple(lab.shape),
        "oracle_pin_max_dlogit": max_d, "oracle_pin_label_mismatch": mism,
    }, os.path.join(out_dir, f"full_{name}.pt"))


EVENT_CASES = {"aott_multi14_events": "aott", "deaott_multi14_events": "deaott"}


def events_case(out_dir, name="aott_multi14_events"):
    """> 10 objects and objects that first appear mid-video, through the reference's AOTInferEngine exactly as
    Evaluator.evaluating drives it (evaluator.py:302-446): 8 objects at frame 0, ids 9..14 annotated at frame 2 (a second
    sub-engine is created there, aot_engine.py:588-594), merged logits from soft_logit_aggregation (:565-582)."""
    model_name, H, W, oh, ow, T, gap = EVENT_CASES[name], 97, 129, 64, 80, 6, 2
    torch.manual_seed(0)
    sd = OW.build_state_dict(model_name, seed=0, flavour="calibrated")
    rcfg = DefaultEngineConfig("golden", model_name)
    ref_model = ref_build_model(rcfg.MODEL_VOS, rcfg).eval()
    ref_model.load_state_dict(sd, strict=True)
    engine = ref_build_engine(rcfg.MODEL_ENGINE, phase="eval", aot_model=ref_model, gpu_id=-1,
                              long_term_mem_gap=gap, short_term_mem_skip=1)
    engine.eval()
    frames, full = O.synthetic_video(T, H, W, 14, seed=4321)
    first = torch.where(full <= 8, full, torch.zeros_like(full))
    new = F.interpolate(torch.where(full > 8, full, torch.zeros_like(full)), size=(oh, ow), mode="nearest")
    with torch.no_grad():
        ref_lo, ref_labels = O.run_video_events(engine, frames, first, 8, (oh, ow), new_objects={2: new})
        oe = O.OracleInferEngine(sd, O.OracleConfig(model_name), long_term_mem_gap=gap)
        o_lo, _ = O.run_video_events(oe, frames, first, 8, (oh, ow), new_objects={2: new}, forced_masks=ref_labels)
    assert [t.shape[1] for t in ref_lo] == [11, 21, 21, 21, 21], [t.shape for t in ref_lo]
    # channels above the live object count hold -1e10-derived values: compare the live ones
    live = [9, 15, 15, 15, 15]
    max_d = max((a[:, :n] - b[:, :n]).abs().max().item() for a, b, n in zip(ref_lo, o_lo, live))
    print(f"[{name}] oracle vs reference: max|dlogit|={max_d:.3e} engines={len(engine.aot_engines)} "
          f"labels used={sorted(set(int(v) for l in ref_labels for v in l.unique().tolist()))}")
    torch.save({
        "model": model_name, "H": H, "W": W, "out_size": (oh, ow), "frames": T, "gap": gap, "seed": 0,
        "video_seed": 4321, "first_objs": 8, "event_frame": 2, "live_channels": live,
        "weights_checksum": OW.checksum(sd), "new_label": new.to(torch.uint8),
        "ref_logits": [t[:, :n].to(torch.float32).clone() for t, n in zip(ref_lo, live)],
        "ref_labels": [t.to(torch.uint8) for t in ref_labels], "oracle_pin_max_dlogit": max_d,
    }, os.path.join(out_dir, f"events_{name}.pt"))


def op_cases(out_dir):
    """Per-op vectors straight from the reference's attention modules (K1, K2, K1', K2')."""
    g = torch.Generator().manual_seed(77)
    out = {}
    with torch.no_grad():
        # K1  MultiheadAttention(use_linear=False)  attention.py:64-121
        m = RA.MultiheadAttention(256, 8, use_linear=False).eval()
        Q = torch.randn(70, 1, 256, generator=g) * 2
        K = torch.randn(333, 1, 256, generator=g)
        V = torch.randn(333, 1, 256, generator=g)
        out["k1"] = {"sd": {k: v.clone() for k, v in m.state_dict().items()}, "Q": Q, "K": K, "V": V,
                     "out": m(Q, K, V)[0]}
        # K3  MultiheadAttention(use_linear=True) (self-attention)
        m = RA.MultiheadAttention(256, 8, use_linear=True).eval()
        X = torch.randn(90, 1, 256, generator=g)
        out["k3"] = {"sd": {k: v.clone() for k, v in m.state_dict().items()}, "X": X, "out": m(X, X, X)[0]}
        # K2  MultiheadLocalAttentionV2 unfold branch  attention.py:308-376
        m = RA.MultiheadLocalAttentionV2(256, 8, use_linear=False, enable_corr=False).eval()
        m.relative_emb_v.data = torch.randn(8, 32, 225, generator=g) * 0.2
        m.relative_emb_k.weight.data = torch.randn(1800, 32, 1, 1, generator=g) * 0.1
        h, w = 9, 20
        q = torch.randn(1, 256, h, w, generator=g)
        k = torch.randn(1, 256, h, w, generator=g)
        v = torch.randn(1, 256, h, w, generator=g)
        o, attn = m(q, k, v)
        out["k2"] = {"sd": {kk: vv.clone() for kk, vv in m.state_dict().items()}, "q": q, "k": k, "v": v,
                     "out": o, "attn": attn}
        # K1' GatedPropagation(use_linear=False)  attention.py:636-712
        m = RA.GatedPropagation(d_qk=64, d_vu=64, num_head=1, use_linear=False, d_att=32).eval()  # small dims: fixture size
        N, Tk, hh, ww = 6 * 7, 150, 6, 7
        Q = torch.randn(N, 1, 32, generator=g) * 2
        K = torch.randn(Tk, 1, 32, generator=g)
        V = torch.randn(Tk, 1, 128, generator=g)
        U = torch.randn(N, 1, 128, generator=g)
        out["k1p"] = {"sd": {kk: vv.clone() for kk, vv in m.state_dict().items()}, "Q": Q, "K": K, "V": V, "U": U,
                      "size_2d": (hh, ww), "out": m(Q, K, V, U, (hh, ww))[0]}
        # K2' LocalGatedPropagation(use_linear=False, enable_corr=False)  attention.py:789-861
        m = RA.LocalGatedPropagation(d_qk=64, d_vu=64, num_head=1, use_linear=False, enable_corr=False,
                                     d_att=32, max_dis=7).eval()
        m.relative_emb_k.weight.data = torch.randn(225, 32, 1, 1, generator=g) * 0.1
        q = torch.randn(1, 32, hh, ww, generator=g)
        k = torch.randn(1, 32, hh, ww, generator=g)
        v = torch.randn(1, 128, hh, ww, generator=g)
        u = torch.randn(N, 1, 128, generator=g)
        out["k2p"] = {"sd": {kk: vv.clone() for kk, vv in m.state_dict().items()}, "q": q, "k": k, "v": v, "u": u,
                      "size_2d": (hh, ww), "out": m(q, k, v, u, (hh, ww))[0]}
        # sine position embedding  position.py:49-74
        from networks.layers.position import PositionEmbeddingSine
        pe = PositionEmbeddingSine(128, normalize=True)
        out["pos"] = {"h": 11, "w": 16, "out": pe(torch.zeros(1, 1, 11, 16))}
    # oracle pin on the op vectors
    W = {"p." + k: v for k, v in out["k1"]["sd"].items()}
    o = O._lin(O.multihead_attention(out["k1"]["Q"], out["k1"]["K"], out["k1"]["V"], 8), W, "p.projection")
    print("[ops] k1 oracle pin", (o - out["k1"]["out"]).abs().max().item())
    c = out["k2"]
    core = O.local_attention(c["q"], c["k"], c["v"], c["sd"]["relative_emb_k.weight"], c["sd"]["relative_emb_k.bias"],
                             c["sd"]["relative_emb_v"], 8)
    o = F.linear(core, c["sd"]["projection.weight"], c["sd"]["projection.bias"])
    print("[ops] k2 oracle pin", (o - c["out"]).abs().max().item())
    c = out["k1p"]
    o, _ = O.gated_propagation({"p." + k: v for k, v in c["sd"].items()}, "p.", c["Q"], c["K"], c["V"], c["U"],
                               c["size_2d"], False)
    print("[ops] k1' oracle pin", (o - c["out"]).abs().max().item())
    c = out["k2p"]
    o, _ = O.local_gated_propagation({"p." + k: v for k, v in c["sd"].items()}, "p.", c["q"], c["k"], c["v"], c["u"],
                                     c["size_2d"])
    print("[ops] k2' oracle pin", (o - c["out"]).abs().max().item())
    print("[ops] pos oracle pin", (O.pos_emb_sine(11, 16) - out["pos"]["out"]).abs().max().item())
    torch.save(out, os.path.join(out_dir, "ops_attention.pt"))


def io_case(out_dir):
    """Row f.3: the reference's own MultiRestrictSize + MultiToTensor (dataloaders/video_transforms.py:594-715) on a seeded
    uint8 frame, and utils.image._save_mask's PNG, as fixtures for the GPU preprocessing kernel and the mask writer."""
    import io as _io
    import numpy as np
    import dataloaders.video_transforms as tr
    import utils.image as RI
    from oracle import io_side as IO
    rng = np.random.default_rng(7)
    small = rng.integers(0, 256, (23, 31, 3)).astype(np.float32)
    img = np.clip(np.kron(small, np.ones((5, 5, 1), np.float32)) + rng.normal(0, 6, (115, 155, 3)), 0, 255).astype(np.uint8)
    cases = {"up_1.3_align": dict(max_short_edge=None, max_long_edge=800, flip=True, multi_scale=[1.0, 1.3], align_corners=True),
             "down_long96": dict(max_short_edge=None, max_long_edge=96, flip=False, multi_scale=[1.0], align_corners=False),
             "short_64": dict(max_short_edge=64, max_long_edge=800, flip=False, multi_scale=[1.0], align_corners=True)}
    out = {"img": torch.from_numpy(img), "cases": {}}
    for name, kw in cases.items():
        sample = {"current_img": np.array(img, dtype=np.float32), "meta": {"flip": False}}
        ref = tr.MultiToTensor()(tr.MultiRestrictSize(kw["max_short_edge"], kw["max_long_edge"], kw["flip"], kw["multi_scale"],
                                                      kw["align_corners"])(sample))
        tensors = [r["current_img"].float().contiguous() for r in ref]
        k, worst = 0, 0.0
        for sc in kw["multi_scale"]:
            for fl in ((False, True) if kw["flip"] else (False,)):
                mine = IO.preprocess(img, kw["max_short_edge"], kw["max_long_edge"], sc, kw["align_corners"], 16, fl)
                worst = max(worst, (mine - tensors[k]).abs().max().item())
                k += 1
        print(f"[io {name}] {[tuple(t.shape) for t in tensors]} oracle vs reference max|d| = {worst:.2e}")
        out["cases"][name] = {"kw": kw, "ref": tensors}
    mask = (rng.integers(0, 4, (20, 27)).astype(np.uint8))
    squeeze = [0, 3, 7, 12]
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        RI._save_mask(mask.copy(), os.path.join(d, "a.png"), None)
        RI._save_mask(mask.copy(), os.path.join(d, "b.png"), squeeze)
        out["mask"] = torch.from_numpy(mask)
        out["squeeze_idx"] = squeeze
        out["png_plain"] = open(os.path.join(d, "a.png"), "rb").read()
        out["png_squeezed"] = open(os.path.join(d, "b.png"), "rb").read()
    torch.save(out, os.path.join(out_dir, "io_side.pt"))


CONTRACT_MODELS = ["aott", "r50_aotl", "deaott", "r50_deaotl", "swinb_aotl", "swinb_deaotl"]


def contract_case(out_dir):
    """What the tests check against the reference without importing it (tests/golden/reference_contract.json.gz): per model
    the state_dict (key -> shape) and the repr of every config value, the DAVIS palette table, and the
    layout of the reference's ``networks`` package with the ``from networks.* import`` statements of each module (the seam
    the overlay package replaces)."""
    import ast
    import gzip
    import json
    import utils.image as RI
    from aot_benchmark_b200 import EngineConfig, build_vos_model
    out = {"models": {}, "palette": list(RI._palette), "networks": {}}
    for m in CONTRACT_MODELS:
        rc, mc = DefaultEngineConfig("x", m), EngineConfig("x", m)
        out["models"][m] = {
            "state_dict": {k: list(v.shape) for k, v in ref_build_model(rc.MODEL_VOS, rc).state_dict().items()},
            "config": {k: repr(v) for k, v in rc.__dict__.items() if k not in ("EXP_NAME", "MODEL_NAME")}}
        b = {k: list(v.shape) for k, v in build_vos_model(mc.MODEL_VOS, mc).state_dict().items()}
        print(f"[contract {m}] {len(b)} parameters, state_dict matches the reference: {b == out['models'][m]['state_dict']}")
    root = os.path.join(REF, "networks")
    for d, _, files in sorted(os.walk(root)):
        for f in sorted(files):
            if f.endswith(".py"):
                path = os.path.join(d, f)
                imports = [[n.module, [a.name for a in n.names]] for n in ast.walk(ast.parse(open(path).read()))
                           if isinstance(n, ast.ImportFrom) and n.module and n.module.split(".")[0] == "networks"]
                out["networks"][os.path.relpath(path, REF)] = imports
    with gzip.GzipFile(os.path.join(out_dir, "reference_contract.json.gz"), "wb", mtime=0) as fh:   # byte-reproducible
        fh.write(json.dumps(out, sort_keys=True).encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "tests", "golden"))
    ap.add_argument("--only", default=None)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    if a.only in (None, "ops"):
        op_cases(a.out)
    for name in VIDEO_CASES:
        if a.only in (None, name):
            video_case(name, a.out)
    for name in EVENT_CASES:
        if a.only in (None, "events", name):
            events_case(a.out, name)
    if a.only == "io":
        io_case(a.out)
    if a.only in (None, "contract"):
        contract_case(a.out)
    for name in FULL_CASES:
        if a.only in ("full", name):              # not part of the default regeneration (minutes of CPU)
            full_case(name, a.out)


if __name__ == "__main__":
    main()
