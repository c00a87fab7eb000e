"""The REFERENCE ITSELF on the GPU next to this engine: the reference's own modules run as infer.py runs them — model.half(),
autocast(fp16), the installed flash-attn — with the restated HF greedy loop (oracle/ref_runner.py), on the same synthetic ArAE weights
and cloud as this repository's CUDA path.  The reference's side is recorded on a B200 in tests/golden/ref_gpu_lmm.npz
(oracle/gen_golden_gpu.py): its 600-token greedy stream, its fp16 logits in full at 48 seeded positions and the 8 best allowed ones at
every position, and its forward-hook dtype ledger.

Asserted: teacher-forced on the reference's stream, |dlogit| mean <= 1.5e-3 / max <= 8e-3 on the fp16 logits HF sees; every id that
differs sits inside the reference's own near-tie band (margin <= 2 * 8e-3 + 1 fp16 ulp); the forward-hook dtype ledger of the reference is
the one oracle mode='ledger' / the kernels implement (SURVEY Appendix B)."""
import json
import os
from dataclasses import replace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_reference_gpu_path_against_engine(golden_dir):
    from core.options import config_defaults
    from edgerunner_b200 import synth
    from edgerunner_b200.engine import Engine
    g = np.load(os.path.join(golden_dir, 'ref_gpu_lmm.npz'))
    ref_tokens = g['tokens'].astype(np.int64)
    T = len(ref_tokens)
    opt = replace(config_defaults['ArAE'], generate_mode='greedy')
    sd = synth.synth_state_dict(opt, seed=0, eos_logit=-30.0)
    cond = synth.synth_point_cloud(0, opt.point_num).to('cuda:0')
    eng = Engine(opt, torch.device('cuda:0'), max_new_tokens=T + 8)
    eng.load_state_dict(sd)
    del sd
    eng.encode_cond(cond[0], 4000)
    eng.prefill([opt.bos_token_id])
    ours = eng.decode(T, mode='greedy', forced=[int(x) for x in ref_tokens], want_logits=True)
    ol16 = ours['logits_pre'].cpu().to(torch.float16).float()
    assert ol16.shape == (T, eng.V)

    rows = torch.as_tensor(g['rows'].astype(np.int64))
    d_rows = (ol16[rows] - torch.as_tensor(g['row_logits']).float()).abs()
    top_ids = torch.as_tensor(g['top_ids'].astype(np.int64))
    top_vals = torch.as_tensor(g['top_vals']).float()
    fin = torch.isfinite(top_vals)                                  # fewer than 8 ids are allowed at some steps
    d_top = (ol16.gather(1, top_ids) - top_vals).abs()[fin]
    tf = {'mean_abs_dlogit': float(d_rows.mean()), 'max_abs_dlogit': max(float(d_rows.max()), float(d_top.max()))}
    mism = np.nonzero(ours['tokens'] != ref_tokens)[0]
    # decision margins of the reference at the mismatching steps (its choice minus ours, in its own fp16 logits)
    margins = []
    for t in mism:
        hit = (top_ids[t] == int(ours['tokens'][t])) & fin[t]
        assert bool(hit.any()), (t, int(ours['tokens'][t]), top_ids[t].tolist())
        margins.append(float(top_vals[t, 0] - top_vals[t][hit][0]))
    tf.update(id_mismatches=int(len(mism)), mismatch_margins_ref_fp16=margins)
    print('reference GPU path vs engine:', json.dumps(tf))
    assert tf['mean_abs_dlogit'] <= 1.5e-3 and tf['max_abs_dlogit'] <= 8e-3, tf
    for m in margins:
        assert m <= 2 * 8e-3 + 0.0079, tf                      # 1 fp16 ulp at |logit| < 8
    assert tf['id_mismatches'] <= T // 100

    led = json.loads(str(g['ledger']))
    # SURVEY Appendix B, observed on the reference: Linear outputs fp16, LayerNorm outputs fp32, embeddings fp16, decode step enters layer 0 in fp16
    for k, v in led.items():
        if "'Linear'" in k:
            assert all(x.endswith('->float16') for x in v), (k, v)
        if "'LayerNorm'" in k:
            assert all(x.endswith('->float32') for x in v), (k, v)
        if "'Embedding'" in k:
            assert all(x.endswith('->float16') for x in v), (k, v)
    assert 'float16->float32' in led["('decode', 'LayerNorm', 'self_attn_layer_norm')"]
    assert str(g['inputs_embeds_dtype']) == 'torch.float32'
