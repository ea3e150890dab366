#!/usr/bin/env python
"""Generates tests/golden/full_width_t2u_ref.npz: what the fp32 oracle (oracle/unity_oracle.py) computes for the bench's
first utterance (seed 1234, 10 s) through seamlessM4T_v2_large with the bench's seeded weights (seed 0, dec_gain 4),
beam 5, hard_max_seq_len 102 - the teacher-forced decoder states of its best hypothesis (in fp16, as the GPU T2U takes
them), the NAR T2U's other inputs, and the units the oracle computes from its fp32 states.

test_full_width_s2st_matches_oracle feeds these states to the GPU T2U and compares unit ids.  The oracle's fp32 states
move by ~1e-4 with the host's thread count and vector ISA, enough to change their fp16 rounding, and three of the 495
units sit at top-1 / top-2 margins below 7e-3, so a comparison against states recomputed on each host would change
with the host.  The fixture fixes them; the test still checks that the live oracle agrees with it.  One thread, so
that regenerating on the same kind of host reproduces the file.

    python tests/golden/make_golden_full_width.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def main():
    from oracle.unity_oracle import UnityOracle, VocoderOracle, s2st
    from seamless_communication_b200 import config as C, synthetic as S
    torch.set_num_threads(1)
    cfg, vc = C.base_v2(), C.base_vocoder()
    toks = S.make_tokenizers(cfg)
    uo = UnityOracle(cfg.to_dict(), S.make_unity_state_dict(cfg, seed=0, dec_gain=4.0), toks)
    vo = VocoderOracle(vc.to_dict(), S.make_vocoder_state_dict(vc, seed=1))
    waves = S.make_waveforms(1, 160000, seed=1234)
    with torch.inference_mode():
        ref = s2st(uo, vo, waves, "spa", 25, 45, hard_max=102)
    n = int(ref["unit_lens"][0])
    top2 = ref["logits"][0, :n].float().topk(2, dim=-1).values
    out = {"dec_out": ref["dec_out"].half().numpy(), "text_seqs": ref["text_seqs"].numpy(), "dur": ref["dur"].numpy(),
           "unit_lens": ref["unit_lens"].numpy(), "units": ref["units"].numpy(),
           "unit_margins": (top2[:, 0] - top2[:, 1]).numpy()}
    np.savez_compressed(os.path.join(HERE, "full_width_t2u_ref.npz"), **out)
    print({k: (v.dtype, v.shape) for k, v in out.items()}, "smallest unit margins", np.sort(out["unit_margins"])[:4])


if __name__ == "__main__":
    main()
