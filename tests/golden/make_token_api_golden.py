"""Generates tests/golden/token_api.json by running the REFERENCE's own implementation of the
task-prompt token API (powerpaint/utils/utils.py of the original project, imported as is with a one-function
`mmengine` stub) on the synthetic CLIP tokenizer / text encoder of synthetic_clip.py.

    PP_REFERENCE_DIR=<checkout of the original PowerPaint project> python tests/golden/make_token_api_golden.py
"""
import importlib.util
import json
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from synthetic_clip import make_text_encoder, make_tokenizer  # noqa: E402

REF = os.path.join(os.environ["PP_REFERENCE_DIR"], "powerpaint", "utils", "utils.py")

PROMPTS = [
    "a photo of a cat P_obj",
    "the dog on the wall P_ctxt",
    "empty scene blur P_shape",
    "P_ctxt a chair P_obj",
    "a photo P_obj P_obj of sky",   # two adjacent runs: exercises the reference's scan quirk
    "a cat",
    "",
]


def load_reference_utils():
    stub = types.ModuleType("mmengine")
    stub.print_log = lambda *a, **k: None
    sys.modules["mmengine"] = stub
    spec = importlib.util.spec_from_file_location("ref_utils", REF)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main():
    ref = load_reference_utils()
    tok_raw = make_tokenizer()
    wrapper = ref.TokenizerWrapper.__new__(ref.TokenizerWrapper)  # __init__ needs from_pretrained (no network)
    wrapper.wrapped = tok_raw
    wrapper._from_pretrained = None
    wrapper.token_map = {}
    te = make_text_encoder(len(tok_raw), seed=0)
    base_vocab = len(tok_raw)
    ref.add_tokens(tokenizer=wrapper, text_encoder=te, placeholder_tokens=["P_ctxt", "P_shape", "P_obj"],
                   initialize_tokens=["a", "a", "a"], num_vectors_per_token=10)
    # distinct, deterministic "learned" vectors (as if loaded from text_encoder.safetensors)
    g = torch.Generator().manual_seed(42)
    emb_layer = te.text_model.embeddings.token_embedding
    with torch.no_grad():
        for name in ["P_ctxt", "P_shape", "P_obj"]:
            emb_layer.trainable_embeddings[name].copy_(torch.randn(10, 32, generator=g))
    out = {"base_vocab": base_vocab, "vocab_after": len(wrapper.wrapped), "token_map": wrapper.token_map,
           "state_dict_keys": sorted(k for k in te.state_dict().keys() if "token_embedding" in k),
           "token_info": {n: wrapper.get_token_info(n) for n in ["P_ctxt", "P_shape", "P_obj"]}, "cases": []}
    for p in PROMPTS:
        enc = wrapper(p, padding="max_length", max_length=77, truncation=True, return_tensors="pt")
        ids = enc.input_ids
        with torch.no_grad():
            tok_emb = emb_layer(ids)          # the spliced token embeddings
            hidden = te(ids)[0]               # full text encoder output
        out["cases"].append({
            "prompt": p,
            "replaced_text": wrapper.replace_placeholder_tokens_in_text(p),
            "input_ids": ids[0].tolist(),
            "token_embedding_sum": tok_emb[0].sum(-1).tolist(),            # per-position checksum
            "token_embedding_first8": tok_emb[0, :, :8].flatten().tolist()[:8 * 20],
            "hidden_sum": hidden[0].sum(-1).tolist(),
            "decode": wrapper.decode(ids[0].tolist(), skip_special_tokens=True),
        })
    with open(os.path.join(HERE, "token_api.json"), "w") as f:
        json.dump(out, f)
    print("wrote token_api.json:", len(out["cases"]), "cases; vocab", base_vocab, "->", out["vocab_after"])


if __name__ == "__main__":
    main()
