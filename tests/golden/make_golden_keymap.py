#!/usr/bin/env python
"""Generates tests/golden/unity_keymap.json by EXECUTING the reference's own checkpoint-conversion functions here
(needs /root/reference; nothing is copied):

  * `_fairseq_key_map`, `convert_unity_checkpoint`, `_get_char_index_mapping`
        (src/seamless_communication/models/unity/loader.py:27-389) and
  * `convert_vocoder_checkpoint` (models/vocoder/loader.py:20-37)

are taken out of their source files with `ast` (the modules import fairseq2, which is absent offline) and run in a
namespace that supplies only what fairseq2 would: a config stand-in with the attributes the functions read for
`unity_archs "base_v2"`, a stand-in character tokenizer, and `convert_fairseq_checkpoint` restated from fairseq2 v0.2
([fs2-recall]: per key, the first pattern whose re.sub changes the key wins).

The input state dict is built FROM the reference's own regex table: one example fairseq key per rule (the pattern with
its groups instantiated), plus the entries the function deletes / rewrites.  The fixture stores old key -> new key and,
for the rewritten tensors, checksums - regenerated deterministically by the test from the same seeds."""
import ast
import json
import math
import os
import re
import sys
import types

import torch

REF = "/root/reference/src/seamless_communication/models"
HERE = os.path.dirname(os.path.abspath(__file__))
CHAR_PIECES = ["<pad>", "<unk>", "<s>", "</s>"] + list("▁etaonzqxm")  # deliberately not sorted


def functions_of(path, names):
    tree = ast.parse(open(path).read())
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in names]
    mod = ast.Module(body=body, type_ignores=[])
    return compile(ast.fix_missing_locations(mod), path, "exec")


def convert_fairseq_checkpoint(checkpoint, key_map):  # fairseq2 v0.2 models/utils/checkpoint.py [fs2-recall]
    def new_key(k):
        for pat, rep in key_map.items():
            n = re.sub(pat, rep, k)
            if n != k:
                return n
        return k
    sd = {new_key(k): v for k, v in checkpoint["model"].items()}
    for k in ("encoder.version", "decoder.version", "encoder.embed_positions._float_tensor", "decoder.embed_positions._float_tensor"):
        sd.pop(k, None)
    return {"model": sd}


class NllbConfig:  # isinstance target
    pass


def base_v2_config():
    nar = types.SimpleNamespace(model_name_or_card="seamlessM4T_v2_large")
    return types.SimpleNamespace(prosody_encoder_config=None, t2u_config=types.SimpleNamespace(nar_decoder_config=nar),
                                 use_text_encoder=True, use_text_decoder=True, use_conformer_adaptor=False,
                                 w2v2_encoder_config=types.SimpleNamespace(use_conformer=True), mt_model_config=NllbConfig())


def char_tokenizer(_name):
    model = types.SimpleNamespace(index_to_token=lambda i: CHAR_PIECES[i], vocabulary_size=len(CHAR_PIECES))
    return types.SimpleNamespace(model=model)


def example_key(pattern):
    k = pattern.lstrip("^").replace("([0-9]+)", "3").replace("(1|2)", "2").replace("\\.", ".")
    return k + ("weight" if k.endswith(".") else "")


def make_inputs(key_map):
    g = torch.Generator().manual_seed(11)
    sd = {}
    for pat in key_map:
        k = example_key(pat)
        sd.setdefault(k, torch.randn(2, 2, generator=g))
    sd["target_letter_decoder.embed_tokens.weight"] = torch.randn(256103, 2, generator=g)
    sd["target_letter_decoder.output_projection.weight"] = sd["target_letter_decoder.embed_tokens.weight"].clone()
    sd["decoder.embed_tokens_text.weight"] = torch.randn(len(CHAR_PIECES), 3, generator=g)
    sd["decoder.embed_tokens_unit.weight"] = torch.randn(12, 3, generator=g)
    sd["decoder.output_projection.weight"] = torch.randn(12, 3, generator=g)
    sd["text_encoder.embed_tokens.weight"] = torch.randn(256103, 2, generator=g)
    for k in ("text_encoder.version", "text_encoder.embed_positions._float_tensor", "target_letter_decoder.version", "target_letter_decoder.embed_positions._float_tensor",
              "encoder.w2v_encoder.w2v_model.mask_emb", "decoder.char_upsampler.embed_positions._float_tensor",
              "decoder.char_upsampler.embed_tokens_char.weight", "decoder.alignment_encoder.conv.weight",
              "decoder_target_letter_decoder.proj.weight", "decoder_target_letter_decoder.proj.bias", "some.unmatched.key"):
        sd[k] = torch.randn(2, generator=g)
    return sd


def checksum(t):
    """Shape, sum and position-weighted sum.  The products are exact in float64 and math.fsum rounds the exact sum, so
    the value does not depend on the order in which a host's torch.sum happens to reduce."""
    v = t.double().flatten()
    return [list(t.shape), math.fsum(v.tolist()), math.fsum((v * torch.arange(1, v.numel() + 1, dtype=torch.float64)).tolist())]


def main():
    ns = {"torch": torch, "Any": object, "Dict": dict, "List": list, "Mapping": dict, "UnitYConfig": object, "NllbConfig": NllbConfig,
          "convert_fairseq_checkpoint": convert_fairseq_checkpoint, "load_unity_char_tokenizer": char_tokenizer}
    exec(functions_of(os.path.join(REF, "unity", "loader.py"), {"convert_unity_checkpoint", "_fairseq_key_map", "_get_char_index_mapping"}), ns)
    cfg = base_v2_config()
    key_map = ns["_fairseq_key_map"](cfg)
    sd_in = make_inputs(key_map)
    rename = {}
    for k in sd_in:  # one key at a time: several fairseq spellings map to the same fairseq2 name
        one = convert_fairseq_checkpoint({"model": {k: 0}}, key_map)["model"]
        rename[k] = next(iter(one)) if one else None
    out = ns["convert_unity_checkpoint"]({"model": {k: v.clone() for k, v in sd_in.items()}}, cfg)["model"]
    vns = {"Any": object, "Mapping": dict, "VocoderConfig": object}
    exec(functions_of(os.path.join(REF, "vocoder", "loader.py"), {"convert_vocoder_checkpoint"}), vns)
    voc = vns["convert_vocoder_checkpoint"]({"generator": {"conv_pre.weight_g": 1, "ups.0.bias": 2}}, None)
    fixture = {"char_pieces": CHAR_PIECES, "patterns": list(key_map.keys()), "rename": rename, "output_keys": sorted(out.keys()),
               "checksums": {k: checksum(out[k]) for k in ("final_proj.weight", "text_decoder_frontend.embed.weight",
                                                           "t2u_model.decoder_frontend.embed_char.weight",
                                                           "t2u_model.decoder_frontend.embed.weight", "t2u_model.final_proj.weight",
                                                           "text_encoder_frontend.embed.weight")},
               "char_index_mapping": ns["_get_char_index_mapping"](cfg), "vocoder_keys": sorted(voc["model"].keys())}
    json.dump(fixture, open(os.path.join(HERE, "unity_keymap.json"), "w"), indent=0)
    print("rules", len(key_map), "input keys", len(sd_in), "output keys", len(out))


if __name__ == "__main__":
    main()
