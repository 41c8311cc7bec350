"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz from the VERBATIM reference.

Needs a checkout of the upstream project:

    PHOTOVERSE_REFERENCE_ROOT=<checkout> python -m oracle.make_golden

For every case in oracle/cases.py this
  1. runs the unmodified reference files (imported by oracle/ref_loader.py) in fp32 and fp64,
  2. runs the oracle restatement on the same deterministic inputs,
  3. asserts oracle == reference (fp64: <= 1e-12 abs; fp32: <= 2e-6 abs), i.e. pins the oracle,
  4. stores the reference's fp64-run outputs (rounded to fp32) as the golden vectors and the
     fp32-run deviation in manifest.json.
It also records the state-dict layout, constructor defaults and constructor errors of the reference classes
(class_layout.json).

Without a checkout, the tests compare the oracle and the CUDA path against these committed outputs.
"""
import json
import os

import numpy as np
import torch

from . import adapter_oracle, cases, ref_loader
from .processor_oracle import dual_branch_attention, fusion_weights, segment_softmax_form

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def run_reference_processor(c: cases.ProcCase, dtype):
    w = cases.proc_weights(c, torch.float64).to(dtype=dtype)
    x, text, img = (t.to(dtype) for t in cases.proc_inputs(c, torch.float64))
    attn, proc = ref_loader.build_reference_layer(w, dtype)
    if (c.w_text, c.w_img) == (1.0, 1.0):
        with torch.no_grad():
            y = attn(x, encoder_hidden_states=(text, img))
    else:
        # grad-enabled stochastic rule (attention_processor.py:413-420): force the branch by
        # controlling the single torch.rand(1) the reference draws from the global CPU RNG.
        want = 0.1 if c.w_img == 0.0 else 0.9
        for seed in range(10000):
            torch.manual_seed(seed)
            u = torch.rand(1).item()
            if abs(u - want) < 0.1:
                break
        torch.manual_seed(seed)
        assert fusion_weights(True, u) == (c.w_text, c.w_img)
        with torch.enable_grad():
            y = attn(x, encoder_hidden_states=(text, img)).detach()
    return y, proc.to_v_ip_norm.detach()


def run_oracle_processor(c: cases.ProcCase, dtype):
    w = cases.proc_weights(c, torch.float64).to(dtype=dtype)
    x, text, img = (t.to(dtype) for t in cases.proc_inputs(c, torch.float64))
    with torch.no_grad():
        return dual_branch_attention(x, text, img, w, c.w_text, c.w_img), \
            segment_softmax_form(x, text, img, w, c.w_text, c.w_img)


def run_reference_adapter(c: cases.AdapterCase, dtype):
    mod = ref_loader.load_reference_adapter_module()
    ad = mod.PhotoVerseAdapter(clip_embedding_dim=1024, cross_attention_dim=768, num_tokens=c.T).to(dtype)
    sd = adapter_oracle.make_state_dict(c.T, c.seed, dtype=torch.float64)
    ad.load_state_dict({k: v.to(dtype) for k, v in sd.items()}, strict=True)
    embs = [e.to(dtype) for e in cases.adapter_inputs(c, torch.float64)]
    with torch.no_grad():
        return ad(embs, token_index=c.token_index)


CTOR_BAD_ARGS = (dict(fusion_rules=(0.5, 0.6)), dict(fusion_rules=[0.5, 0.5]), dict(scale=[1.0, 2.0]))


def class_layout(processor_cls, adapter_cls):
    """What a checkpoint or a caller sees of a processor / adapter class pair (attention_processor.py:27-56,
    adapters.py:14-28): state-dict shapes and key order, constructor defaults (repr keeps their types) and the texts of
    the constructor's ValueErrors (None where a bad argument is not rejected)."""
    p = processor_cls(hidden_size=320, cross_attention_dim=768, num_tokens=(5,))
    errors = []
    for bad in CTOR_BAD_ARGS:
        try:
            processor_cls(320, 768, **bad)
            errors.append(None)
        except ValueError as e:
            errors.append(str(e))
    return {"processor_state_dict": [[k, list(v.shape)] for k, v in p.state_dict().items()],
            "processor_defaults": repr((p.scale, p.fusion_rule1, p.fusion_rule2, p.num_tokens)),
            "processor_ctor_errors": errors,
            "adapter_state_dict_keys": list(adapter_cls(num_tokens=3).state_dict().keys())}


def main():
    assert ref_loader.reference_available(), "set PHOTOVERSE_REFERENCE_ROOT to a checkout of the upstream project"
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    manifest = {"generator": "oracle/make_golden.py", "torch": torch.__version__, "cases": {}}
    torch.set_num_threads(8)

    for c in cases.PROC_CASES:
        out = {}
        for dtype, tag, tol in ((torch.float64, "f64", 1e-12), (torch.float32, "f32", 2e-6)):
            y_ref, n_ref = run_reference_processor(c, dtype)
            (y_or, n_or), (y_seg, n_seg) = run_oracle_processor(c, dtype)
            e_y = (y_or - y_ref).abs().max().item()
            e_n = (n_or - n_ref).abs().max().item()
            e_seg = (y_seg - y_ref).abs().max().item()
            assert e_y <= tol and e_n <= tol, (c.name, tag, e_y, e_n)
            assert e_seg <= tol * 10 and (n_seg - n_ref).abs().max().item() <= tol * 10, (c.name, tag, e_seg)
            out[f"y_{tag}"] = y_ref.numpy()
            out[f"vnorm_{tag}"] = n_ref.numpy()
            print(f"{c.name:32s} {tag}: oracle-ref {e_y:.2e}  vnorm {e_n:.2e}  segment-form-ref {e_seg:.2e}")
        e32 = np.abs(out["y_f32"].astype(np.float64) - out["y_f64"]).max()
        manifest["cases"][c.name] = {"kind": "processor", "ref_f32_vs_f64_maxabs": float(e32),
                                     "y_rms": float(np.sqrt((out["y_f64"] ** 2).mean()))}
        # keep fixtures small: store the reference's fp64 run rounded to fp32 (<= 6e-8 relative,
        # far below every tolerance used); the fp32-run deviation is recorded in the manifest.
        np.savez_compressed(os.path.join(GOLDEN_DIR, c.name + ".npz"),
                            y=out["y_f64"].astype(np.float32), vnorm=out["vnorm_f64"].astype(np.float32))

    for c in cases.ADAPTER_CASES:
        out = {}
        sd64 = adapter_oracle.make_state_dict(c.T, c.seed, dtype=torch.float64)
        for dtype, tag, tol in ((torch.float64, "f64", 1e-11), (torch.float32, "f32", 2e-5)):
            y_ref = run_reference_adapter(c, dtype)
            embs = [e.to(dtype) for e in cases.adapter_inputs(c, torch.float64)]
            with torch.no_grad():
                y_or = adapter_oracle.adapter_forward(embs, {k: v.to(dtype) for k, v in sd64.items()}, c.token_index)
            e = (y_or - y_ref).abs().max().item()
            assert e <= tol, (c.name, tag, e)
            out[f"y_{tag}"] = y_ref.numpy()
            print(f"{c.name:32s} {tag}: oracle-ref {e:.2e}")
        manifest["cases"][c.name] = {"kind": "adapter",
                                     "ref_f32_vs_f64_maxabs": float(np.abs(out["y_f32"] - out["y_f64"]).max()),
                                     "y_rms": float(np.sqrt((out["y_f64"] ** 2).mean()))}
        np.savez_compressed(os.path.join(GOLDEN_DIR, c.name + ".npz"), y=out["y_f64"].astype(np.float32))

    # concept-token injection (models/clip.py:17-24): the verbatim function is compiled from the reference source
    from . import clip_oracle
    fn = ref_loader.load_reference_inject_fn()
    x, cpt, idx = clip_oracle.inject_case()
    ref = fn(x, cpt, idx)
    assert torch.equal(ref, clip_oracle.inject_concept_embeddings(x, cpt, idx)), "inject oracle != reference"
    np.savez_compressed(os.path.join(GOLDEN_DIR, "inject_concept.npz"), y=ref.numpy()[:, :, :32].copy(), idx=np.array(idx))
    manifest["cases"]["inject_concept"] = {"kind": "inject", "note": "verbatim models/clip.py:_inject_concept_embeddings, "
                                                                     "first 32 of 768 channels stored"}
    print("inject_concept                   : oracle == reference (bit exact)")

    layout = class_layout(ref_loader.load_reference_processor_module().PhotoVerseAttnProcessor2_0,
                          ref_loader.load_reference_adapter_module().PhotoVerseAdapter)
    with open(os.path.join(GOLDEN_DIR, "class_layout.json"), "w") as f:
        json.dump({"provenance": "upstream classes, written by oracle/make_golden.py", "layout": layout}, f, indent=1)

    with open(os.path.join(GOLDEN_DIR, "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1, sort_keys=True)
    print("wrote", GOLDEN_DIR)


if __name__ == "__main__":
    main()
