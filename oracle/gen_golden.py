"""Generate golden vectors by EXECUTING THE REFERENCE (build container only; needs /root/reference).

TEST INFRASTRUCTURE.  Run as a standalone process:  ``python oracle/gen_golden.py [--only tiny|arae|meto|meta|provider|train]``

The reference modules (``core.models.LMM``, ``core.transformer.*``) are imported from /root/reference
with ``flash_attn`` masked (so ``core/transformer/attention.py:19-25`` picks its naive bmm path on CPU)
and with import-time stubs for packages that are absent here and never touched by the arithmetic
(``kiui``, ``trimesh``, ``megfile``).  ``LMM.generate`` itself runs unmodified (FSM closure, kwargs,
``save_mesh`` tail); only ``mesh_decoder.generate`` — third-party HF ``GenerationMixin`` code that the
installed transformers 5.5 cannot run against the reference's tuple cache (``modeling_opt.py:524``) — is
replaced by ``hf_sample_restated`` below, a restatement of transformers==4.46.2 ``_sample``.

Weights are ``edgerunner_b200.synth.synth_state_dict`` loaded with ``load_state_dict(strict=True)``: this
also pins ``state_dict_spec`` against the reference's key schema and shapes.
Outputs: small ``.npz`` / ``.json`` files under tests/golden/ (committed).
"""

import argparse
import dataclasses
import json
import math
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
REF = '/root/reference'
GOLD = os.path.join(REPO, 'tests', 'golden')


def install_stubs():
    sys.modules['flash_attn'] = None  # force the naive attention path (CPU)

    kiui = types.ModuleType('kiui')
    kiui.lo = lambda *a, **k: None
    kiui.seed_everything = lambda s: (torch.manual_seed(s), np.random.seed(s))
    mu = types.ModuleType('kiui.mesh_utils')
    mu.clean_mesh = mu.decimate_mesh = lambda *a, **k: (_ for _ in ()).throw(NotImplementedError)
    op = types.ModuleType('kiui.op')
    op.recenter = lambda *a, **k: (_ for _ in ()).throw(NotImplementedError)
    kiui.mesh_utils, kiui.op = mu, op
    sys.modules.update({'kiui': kiui, 'kiui.mesh_utils': mu, 'kiui.op': op})

    tm = types.ModuleType('trimesh')

    class Trimesh:  # holder only: the cleanup calls are third-party trimesh (parity unpinned, SURVEY §8c)
        def __init__(self, vertices=None, faces=None, **k):
            self.vertices, self.faces = np.asarray(vertices), np.asarray(faces)

        def merge_vertices(self): pass
        def unique_faces(self): return np.ones(len(self.faces), dtype=bool)
        def update_faces(self, m): pass
        def fix_normals(self): pass

    tm.Trimesh = Trimesh
    sys.modules['trimesh'] = tm
    sys.modules['megfile'] = types.ModuleType('megfile')


def import_reference():
    install_stubs()
    # our repo's edgerunner_b200 (synth) + the reference's `core` / `meto` packages; NOT our own `core`
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or '.') != REPO]
    sys.path.insert(0, os.path.join(REF, 'meto'))
    sys.path.insert(0, os.path.join(HERE, '_ref'))      # compiled reference _meto
    sys.path.insert(0, REF)
    import importlib.util
    spec = importlib.util.spec_from_file_location('er_synth', os.path.join(REPO, 'edgerunner_b200', 'synth.py'))
    synth = importlib.util.module_from_spec(spec)
    # synth imports core.options lazily only in tiny_options(); give it the reference's (identical fields)
    spec.loader.exec_module(synth)
    return synth


def hf_sample_restated(decoder, inputs_embeds, eos_token_id, max_new_tokens, prefix_allowed_tokens_fn,
                       do_sample=False, top_k=None, record=None, **unused):
    """transformers==4.46.2 ``GenerationMixin._sample`` for B==1, num_beams==1, inputs_embeds-only prompt.

    input_ids starts as an empty [1,0] long tensor; per step: prepare_inputs_for_generation -> forward ->
    ``logits[:, -1, :].float()`` -> PrefixConstrainedLogitsProcessor (patched: core/utils.py:143-158) ->
    [TopKLogitsWarper(top_k, filter=-inf, min_tokens_to_keep=1)] -> softmax+multinomial | argmax -> append ->
    stop on EOS or len == max_new_tokens.  Returns only the new tokens."""
    B = inputs_embeds.shape[0]
    assert B == 1
    input_ids = torch.ones((B, 0), dtype=torch.long)
    past = None
    attention_mask = torch.ones(inputs_embeds.shape[:2], dtype=torch.long)
    while True:
        mi = decoder.prepare_inputs_for_generation(input_ids, past_key_values=past, attention_mask=attention_mask,
                                                   inputs_embeds=inputs_embeds, use_cache=True)
        out = decoder(**mi, return_dict=True)
        past = out.past_key_values
        logits = out.logits[:, -1, :].clone().float()
        mask = torch.full_like(logits, -math.inf)
        allowed = prefix_allowed_tokens_fn(0, input_ids[0])
        assert len(allowed) > 0
        mask[0, allowed] = 0
        scores = logits + mask
        if do_sample:
            k = min(top_k, scores.size(-1))
            remove = scores < torch.topk(scores, k)[0][..., -1, None]
            scores = scores.masked_fill(remove, -float('inf'))
            probs = torch.softmax(scores, dim=-1)
            nxt = torch.multinomial(probs, num_samples=1).squeeze(1)
        else:
            nxt = torch.argmax(scores, dim=-1)
        if record is not None:
            record['logits'].append(out.logits[0, -1].detach().clone())
            record['scores'].append(scores[0].clone())
        input_ids = torch.cat([input_ids, nxt[:, None]], dim=-1)
        attention_mask = torch.cat([attention_mask, attention_mask.new_ones((B, 1))], dim=-1)
        if int(nxt) == eos_token_id or input_ids.shape[1] >= max_new_tokens:
            return input_ids


def build_reference_model(synth, opt, seed, eos_logit):
    from core.models import LMM
    torch.manual_seed(0)
    model = LMM(opt).eval()
    sd = synth.synth_state_dict(opt, seed=seed, eos_logit=eos_logit)
    ref_sd = model.state_dict()
    assert list(ref_sd.keys()) == [n for n, _, _ in synth.state_dict_spec(opt)] or set(ref_sd) == set(sd), \
        (set(ref_sd) ^ set(sd))
    for k in ref_sd:
        assert tuple(ref_sd[k].shape) == tuple(sd[k].shape), (k, ref_sd[k].shape, sd[k].shape)
    model.load_state_dict(sd, strict=True)
    return model, sd


class RefTokenizer:
    """meto.Engine surface backed by the compiled reference _meto (meto/meto/__init__.py:21-50)."""

    def __init__(self, bins):
        import _meto
        self.impl = _meto.Engine_LR_ABSCO(bins, False)

    def decode(self, tokens):
        v, f, t = self.impl.decode(list(map(int, tokens)))
        return np.asarray(v), np.asarray(f), np.asarray(t)


def run_generate(model, opt, cond, num_faces, max_new, mode, seed=None):
    record = {'logits': [], 'scores': []}

    def fake_generate(**kw):
        return hf_sample_restated(model.mesh_decoder, kw['inputs_embeds'], kw['eos_token_id'], kw['max_new_tokens'],
                                  kw['prefix_allowed_tokens_fn'], do_sample=kw.get('do_sample', False),
                                  top_k=kw.get('top_k'), record=record)

    model.mesh_decoder.generate = fake_generate
    model.opt.generate_mode = mode
    if seed is not None:
        torch.manual_seed(seed)
    with torch.no_grad():
        meshes, toks = model.generate(cond, num_faces=num_faces, max_new_tokens=max_new,
                                      tokenizer=RefTokenizer(opt.discrete_bins), clean=True)
    return toks[0], torch.stack(record['logits']).numpy(), torch.stack(record['scores']).numpy(), meshes[0]


def gen_model_goldens(synth, name, opt, steps, num_faces, sample_steps=0, tf_len=0):
    print(f'[gen] {name}: building reference LMM ...', flush=True)
    model, sd = build_reference_model(synth, opt, seed=0, eos_logit=-30.0)
    cond = synth.synth_point_cloud(seed=0, n=opt.point_num)
    out = {}
    with torch.no_grad():
        post = model.point_encoder(cond)
        out['latents'] = post.mode()[0].numpy()
        ce = model.encode_cond(cond, torch.full((1,), num_faces, dtype=torch.long))['cond_embeds'][0].numpy()
    out['cond_embeds_head'] = ce[:4]
    out['cond_embeds_tail'] = ce[-2:]
    out['cond_embeds_sum'] = ce.astype(np.float64).sum(0)
    toks, logits, scores, mesh = run_generate(model, opt, cond, num_faces, steps, 'greedy')
    out['greedy_tokens'] = toks
    out['greedy_logits'] = logits
    out['mesh_vertices'] = mesh.vertices
    out['mesh_faces'] = mesh.faces
    print(f'[gen] {name}: greedy tokens[:16] = {toks[:16]}', flush=True)
    if sample_steps:
        toks, logits, scores, _ = run_generate(model, opt, cond, num_faces, sample_steps, 'sample', seed=1234)
        out['sample_tokens'] = toks
        out['sample_logits'] = logits
    if tf_len:
        # teacher-forced forward (core/models.py:147-202) on grammar-valid random tokens, dense causal
        B = 2
        rng = np.random.RandomState(7)
        body = grammar_tokens(rng, tf_len, opt.discrete_bins)
        toks_tf = np.stack([np.concatenate([[1], np.roll(body, 4 * b), [2]]) for b in range(B)])
        P = opt.num_cond_tokens
        labels = np.concatenate([np.full((B, P + 1), -100), toks_tf[:, 1:]], axis=1)
        conds = torch.cat([synth.synth_point_cloud(seed=b, n=opt.point_num) for b in range(B)])
        data = dict(conds=conds, tokens=torch.from_numpy(toks_tf).long(), labels=torch.from_numpy(labels).long(),
                    masks=torch.ones(labels.shape, dtype=torch.bool), num_faces=torch.tensor([num_faces, 2500]),
                    num_tokens=torch.tensor([tf_len, tf_len]))
        with torch.no_grad():
            res = model(data)
        out['tf_tokens'] = toks_tf
        out['tf_labels'] = labels
        out['tf_num_faces'] = np.array([num_faces, 2500])
        out['tf_loss'] = np.array([float(res['loss']), float(res['loss_ce']), float(res['loss_kl'])])
        out['tf_logits_tail'] = res['logits'][:, -8:].numpy()
    np.savez_compressed(os.path.join(GOLD, name + '.npz'), **out)
    print(f'[gen] wrote {name}.npz', flush=True)


def train_probe_indices(numel, k=48):
    """the positions of a gradient tensor the training fixture records (shared with tests/test_train_cpu.py)"""
    return np.unique(np.linspace(0, numel - 1, num=min(k, numel)).astype(np.int64))


def gen_train_goldens(synth):
    """The REFERENCE's own training step on the CPU (fp32, naive attention): ``model.train(); out = model(data); out['loss'].backward()``
    (main.py:160-172) for the tiny preset in cond_mode 'point' (the reference always trains the point encoder there: models.py:54 asserts
    ``not opt.freeze_encoder``) and 'point_latent' (no encoder, conds = latents).  Stochastic parts are
    switched off so that the gradients are a function of the inputs alone: config.dropout = 0, nof_dropout_ratio = 0; opt.checkpointing = False
    (same arithmetic, no torch.utils.checkpoint).  Recorded per parameter: the gradient's L2 norm and probe values at fixed positions."""
    out = {}
    for tag, cond_mode in (('point', 'point'), ('latent', 'point_latent')):
        opt = synth.tiny_options(cond_mode=cond_mode, freeze_encoder=False, nof_dropout_ratio=0.0, checkpointing=False, kl_weight=3e-3)
        model, sd = build_reference_model(synth, opt, seed=0, eos_logit=-30.0)
        model.config.dropout = 0.0
        assert all(l.config.dropout == 0.0 for l in model.mesh_decoder.model.layers)
        model.train()
        B, tf_len, num_faces = 2, 40, 1000
        rng = np.random.RandomState(11)
        body = grammar_tokens(rng, tf_len, opt.discrete_bins)
        toks_tf = np.stack([np.concatenate([[1], np.roll(body, 4 * b), [2]]) for b in range(B)])
        P = opt.num_cond_tokens
        labels = np.concatenate([np.full((B, P + 1), -100), toks_tf[:, 1:]], axis=1)
        if cond_mode == 'point':
            conds = torch.cat([synth.synth_point_cloud(seed=b, n=opt.point_num) for b in range(B)])
        else:
            conds = torch.randn(B, opt.point_latent_size, opt.point_latent_dim, generator=torch.Generator().manual_seed(5)) * 0.5
            out['latent_conds'] = conds.numpy()
        data = dict(conds=conds, tokens=torch.from_numpy(toks_tf).long(), labels=torch.from_numpy(labels).long(),
                    masks=torch.ones(labels.shape, dtype=torch.bool), num_faces=torch.tensor([num_faces, 2500]),
                    num_tokens=torch.tensor([tf_len, tf_len]))
        res = model(data)
        res['loss'].backward()
        out[f'{tag}_loss'] = np.array([float(res['loss']), float(res['loss_ce']), float(res.get('loss_kl', 0.0))])
        names = []
        for n, p in model.named_parameters():
            if p.grad is None:
                continue
            g = p.grad.detach().double().reshape(-1).numpy()
            names.append(n)
            out[f'{tag}|{n}|norm'] = np.array(np.linalg.norm(g))
            out[f'{tag}|{n}|probe'] = g[train_probe_indices(g.size)].astype(np.float32)
        out[f'{tag}_names'] = np.array(names)
        print(f'[gen] train/{tag}: loss {float(res["loss"]):.6f}, {len(names)} tensors with gradients', flush=True)
        if tag == 'point':
            out['tokens'], out['labels'], out['num_faces'] = toks_tf, labels, np.array([num_faces, 2500])
    np.savez_compressed(os.path.join(GOLD, 'train.npz'), **out)
    print('[gen] wrote train.npz', flush=True)


def grammar_tokens(rng, n, bins):
    """Random FSM-valid stream (BOM + 9 coords, then L/R + 3 coords ...), already +3 offset, length n."""
    t = [5] + list(rng.randint(6, 6 + bins, size=9))
    while len(t) + 4 <= n:
        if rng.rand() < 0.05 and len(t) + 10 <= n:
            t += [5] + list(rng.randint(6, 6 + bins, size=9))
        else:
            t += [int(rng.choice([3, 4]))] + list(rng.randint(6, 6 + bins, size=3))
    while len(t) < n:
        t.append(int(rng.randint(6, 6 + bins)))
    return np.asarray(t[:n], dtype=np.int64)


def fixture_meshes():
    """The inline meshes of /root/reference/meto/tests/engine.py:39-118 are rebuilt procedurally here in
    tests/meshes.py (shared with the tests); sphere/annulus need trimesh (absent) and are replaced by an
    icosphere / annulus generated by our own code."""
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import meshes
    return meshes.all_meshes()


def gen_meto_goldens():
    import _meto
    out = {}
    names = []
    for name, (v, f) in fixture_meshes().items():
        for bins in (512, 2048):
            eng = _meto.Engine_LR_ABSCO(bins, False)
            tok, order, ftype = eng.encode(v.astype(np.float32).tolist(), f.astype(np.int32).tolist())
            dv, df, dt = eng.decode(tok)
            key = f'{name}_{bins}'
            names.append(key)
            out[key + '_tokens'] = np.asarray(tok, dtype=np.int32)
            out[key + '_order'] = np.asarray(order, dtype=np.int32)
            out[key + '_ftype'] = np.asarray(ftype, dtype=np.int32)
            out[key + '_dv'] = np.asarray(dv, dtype=np.float64).reshape(-1, 3)
            out[key + '_df'] = np.asarray(df, dtype=np.int32).reshape(-1, 3)
            out[key + '_dt'] = np.asarray(dt, dtype=np.int32)
    # encode-only stress cases (coarse bins force ties between face centres and coincident quantised vertices)
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import meshes
    enc_names = []
    for name, (v, f) in meshes.stress_meshes().items():
        for bins in (8, 64, 512):
            eng = _meto.Engine_LR_ABSCO(bins, False)
            tok, order, ftype = eng.encode(v.astype(np.float32).tolist(), f.astype(np.int32).tolist())
            key = f'{name}_{bins}'
            enc_names.append(key)
            out[key + '_tokens'] = np.asarray(tok, dtype=np.int16)
            out[key + '_order'] = np.asarray(order, dtype=np.int16)
            out[key + '_ftype'] = np.asarray(ftype, dtype=np.int8)
    out['enc_names'] = np.asarray(enc_names)
    # random / malformed streams for the decoder (truncations, coord where an op is expected, empty)
    rng = np.random.RandomState(11)
    streams = [np.zeros(0, np.int64), grammar_tokens(rng, 4001, 512) - 3, grammar_tokens(rng, 57, 512) - 3,
               grammar_tokens(rng, 9, 512) - 3, grammar_tokens(rng, 10, 512) - 3, grammar_tokens(rng, 12, 512) - 3]
    bad = grammar_tokens(rng, 200, 512) - 3
    bad[50] = 300  # make sure something breaks the op/coord alternation somewhere
    streams.append(bad)
    eng = _meto.Engine_LR_ABSCO(512, False)
    for i, s in enumerate(streams):
        dv, df, dt = eng.decode([int(x) for x in s])
        out[f'stream{i}_tokens'] = s.astype(np.int32)
        out[f'stream{i}_dv'] = np.asarray(dv, dtype=np.float64).reshape(-1, 3)
        out[f'stream{i}_df'] = np.asarray(df, dtype=np.int32).reshape(-1, 3)
        out[f'stream{i}_dt'] = np.asarray(dt, dtype=np.int32)
    # ---- LR backend (Options.meto_backend = 'LR'): encode + decode of the fixtures, encode of the stress meshes, malformed streams ----
    lr_names, lr_enc_names = [], []
    for name, (v, f) in fixture_meshes().items():
        eng = _meto.Engine_LR(512, False)
        tok, order, ftype = eng.encode(v.astype(np.float32).tolist(), f.astype(np.int32).tolist())
        dv, df, dt = eng.decode(tok)
        key = f'lr_{name}_512'
        lr_names.append(key)
        out[key + '_tokens'] = np.asarray(tok, dtype=np.int32)
        out[key + '_order'] = np.asarray(order, dtype=np.int32)
        out[key + '_ftype'] = np.asarray(ftype, dtype=np.int32)
        out[key + '_dv'] = np.asarray(dv, dtype=np.float64).reshape(-1, 3)
        out[key + '_df'] = np.asarray(df, dtype=np.int32).reshape(-1, 3)
        out[key + '_dt'] = np.asarray(dt, dtype=np.int32)
    for name, (v, f) in meshes.stress_meshes().items():
        for bins in (8, 512):
            tok, order, ftype = _meto.Engine_LR(bins, False).encode(v.astype(np.float32).tolist(), f.astype(np.int32).tolist())
            key = f'lr_{name}_{bins}'
            lr_enc_names.append(key)
            out[key + '_tokens'] = np.asarray(tok, dtype=np.int16)
            out[key + '_order'] = np.asarray(order, dtype=np.int16)
            out[key + '_ftype'] = np.asarray(ftype, dtype=np.int8)
    rng = np.random.RandomState(12)
    lr_streams = [np.zeros(0, np.int64), grammar_tokens(rng, 2001, 1024) - 3, grammar_tokens(rng, 10, 1024) - 3, grammar_tokens(rng, 11, 1024) - 3]
    bad = grammar_tokens(rng, 120, 1024) - 3
    bad[40] = 900; bad[77] = -1
    lr_streams.append(bad)
    eng = _meto.Engine_LR(512, False)
    for i, s in enumerate(lr_streams):
        dv, df, dt = eng.decode([int(x) for x in s])
        out[f'lr_stream{i}_tokens'] = s.astype(np.int32)
        out[f'lr_stream{i}_dv'] = np.asarray(dv, dtype=np.float64).reshape(-1, 3)
        out[f'lr_stream{i}_df'] = np.asarray(df, dtype=np.int32).reshape(-1, 3)
        out[f'lr_stream{i}_dt'] = np.asarray(dt, dtype=np.int32)
    out['lr_names'] = np.asarray(lr_names)
    out['lr_enc_names'] = np.asarray(lr_enc_names)
    out['n_lr_streams'] = np.asarray(len(lr_streams))
    out['names'] = np.asarray(names)
    out['n_streams'] = np.asarray(len(streams))
    np.savez_compressed(os.path.join(GOLD, 'meto.npz'), **out)
    print('[gen] wrote meto.npz', flush=True)


def clers_op_positions(tok):
    """Indices of the operator tokens of a well-formed Engine_CLERS stream (BOM + 9 coordinates, op, (3 coordinates, op)*, EOM)."""
    pos, i = [], 0
    while i < len(tok):
        if tok[i] == 5:
            i += 10
        elif tok[i] == 6:
            i += 1
        else:
            pos.append(i)
            i += 1 if (i + 1 < len(tok) and tok[i + 1] in (5, 6)) or tok[i] == 2 and i + 1 < len(tok) and tok[i + 1] == 6 else 4
    return pos


def gen_meto_clers_goldens():
    """Engine_CLERS (meto/include/meto/engine_clers.h): encode + decode of the fixtures and stress meshes, and truncated / corrupted streams.
    Streams on which the reference itself reads out of bounds (an E as the very last token, an E that pops an empty stack) are left out."""
    import _meto
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import meshes
    out, names = {}, []
    fx = dict(fixture_meshes())
    cases = [(n, b) for n in fx for b in (512,)] + [(n, b) for n in meshes.stress_meshes() for b in (8, 512)]
    fx.update(meshes.stress_meshes())
    for name, bins in cases:
        v, f = fx[name]
        eng = _meto.Engine_CLERS(bins, False)
        tok, order, ftype = eng.encode(v.astype(np.float32).tolist(), f.astype(np.int32).tolist())
        dv, df, dt = eng.decode(tok)
        key = f'clers_{name}_{bins}'
        names.append(key)
        out[key + '_tokens'] = np.asarray(tok, dtype=np.int16 if 4 * bins + 7 < 32768 else np.int32)
        out[key + '_order'] = np.asarray(order, dtype=np.int32)
        out[key + '_ftype'] = np.asarray(ftype, dtype=np.int8)
        out[key + '_dv'] = np.asarray(dv, dtype=np.float32).reshape(-1, 3)
        out[key + '_df'] = np.asarray(df, dtype=np.int32).reshape(-1, 3)
        out[key + '_dt'] = np.asarray(dt, dtype=np.int8)
    # truncations of one stream at every length (minus the out-of-bounds ones), and coordinates where an operator is expected
    v, f = fx['two_components']
    eng = _meto.Engine_CLERS(64, False)
    tok = list(eng.encode(v.astype(np.float32).tolist(), f.astype(np.int32).tolist())[0])
    ops = set(clers_op_positions(tok))
    streams = [[]]
    for n in range(1, min(len(tok), 160)):
        if (n - 1) in ops and tok[n - 1] == 2:
            continue
        streams.append(tok[:n])
    rng = np.random.RandomState(13)
    for _ in range(6):
        bad = list(tok)
        k = sorted(ops)[rng.randint(1, len(ops) - 1)]
        if bad[k] == 2:
            continue
        bad[k] = 7 + rng.randint(0, 4 * 64)
        streams.append(bad)
    for i, s in enumerate(streams):
        dv, df, dt = eng.decode([int(x) for x in s])
        out[f'clers_stream{i}_tokens'] = np.asarray(s, dtype=np.int16)
        out[f'clers_stream{i}_dv'] = np.asarray(dv, dtype=np.float32).reshape(-1, 3)
        out[f'clers_stream{i}_df'] = np.asarray(df, dtype=np.int16).reshape(-1, 3)
        out[f'clers_stream{i}_dt'] = np.asarray(dt, dtype=np.int8)
    out['names'] = np.asarray(names)
    out['n_streams'] = np.asarray(len(streams))
    np.savez_compressed(os.path.join(GOLD, 'meto_clers.npz'), **out)
    print('[gen] wrote meto_clers.npz', len(names), 'meshes', len(streams), 'streams', flush=True)


def gen_meto_live_goldens():
    """The compiled reference's Engine_LR_ABSCO / Engine_LR on meshes.random_grids(): encode, then decode of its own tokens.  Each field
    of all encodings is stored concatenated (in the dtype that holds it exactly: the decoded vertices are fp32 values) with a length per
    encoding, in iteration order, LR_ABSCO before LR."""
    import _meto
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import meshes
    fields = {'tokens': np.int16, 'order': np.int16, 'ftype': np.int8, 'dv': np.float32, 'df': np.int16, 'dt': np.int8}
    parts = {k: [] for k in fields}
    bins_all = []
    for it, v, f, bins in meshes.random_grids():
        for ref_cls in (_meto.Engine_LR_ABSCO, _meto.Engine_LR):
            ref = ref_cls(bins, False)
            tok, order, ftype = ref.encode(v.tolist(), f.tolist())
            dv, df, dt = ref.decode(tok)
            got = {'tokens': tok, 'order': order, 'ftype': ftype, 'dv': np.reshape(dv, (-1, 3)), 'df': np.reshape(df, (-1, 3)), 'dt': dt}
            for k, dtype in fields.items():
                a = np.asarray(got[k])
                assert np.array_equal(a.astype(dtype), a), k
                parts[k].append(a.astype(dtype))
            bins_all.append(bins)
    out = {'bins': np.asarray(bins_all, dtype=np.int32)}
    for k, p in parts.items():
        out[k] = np.concatenate(p)
        out['n_' + k] = np.asarray([len(x) for x in p], dtype=np.int32)
    np.savez_compressed(os.path.join(GOLD, 'meto_live.npz'), **out)
    print('[gen] wrote meto_live.npz', len(bins_all), 'encodings', flush=True)


def gen_dit_goldens():
    """The reference DiT module itself (core/transformer/dit.py), CPU fp32, naive attention, on the seeded weights of oracle/dit_oracle.py."""
    from core.transformer.dit import DiT
    sys.path.insert(0, HERE)
    from dit_oracle import synth_dit_state
    cfg = dict(hidden_dim=128, num_heads=2, latent_size=40, latent_dim=16, num_layers=2)
    sd = synth_dit_state(**cfg, seed=3)
    m = DiT(**cfg, gradient_checkpointing=False).eval()
    missing, unexpected = m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, cfg['latent_size'], cfg['latent_dim'], generator=g)
    c = torch.randn(2, 9, cfg['hidden_dim'], generator=g)
    t = torch.tensor([991.0, 3.0])
    with torch.no_grad():
        out = m(x, c, t)
    keys = sorted(m.state_dict().keys())
    np.savez_compressed(os.path.join(GOLD, 'dit.npz'), x=x.numpy(), c=c.numpy(), t=t.numpy(), out=out.numpy(), keys=np.asarray(keys),
                        shapes=np.asarray([','.join(map(str, m.state_dict()[k].shape)) for k in keys]), cfg=json.dumps(cfg))
    print('[gen] wrote dit.npz', float(out.abs().mean()), flush=True)


def gen_meta(synth):
    from core.options import config_defaults
    from core.models import LMM
    meta = {'options': {k: dataclasses.asdict(v) for k, v in config_defaults.items()}}
    with open(os.path.join(GOLD, 'options.json'), 'w') as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    from core.utils import quantize_num_faces
    q = {str(n): int(quantize_num_faces(n)) for n in (-1, 0, 1, 999, 1000, 1001, 2000, 2001, 4000, 4001, 8000, 8001, 10 ** 6)}
    with open(os.path.join(GOLD, 'quantize_num_faces.json'), 'w') as f:
        json.dump(q, f)
    print('[gen] wrote options.json / quantize_num_faces.json', flush=True)


def provider_items(rng, opt, lens):
    """Synthetic dataset items with the reference's keys (provider.py:437-466): deterministic per call order."""
    items = []
    for i, n in enumerate(lens):
        items.append(dict(cond=rng.uniform(-0.95, 0.95, (opt.point_num, 3)).astype(np.float32),
                          coords=rng.randint(3, opt.discrete_bins + 3, size=n).astype(np.int64), len=int(n),
                          num_faces=int(rng.randint(10, 9000)), azimuth=int(rng.randint(0, 360)), path=f'item{i}'))
    return items


def gen_provider_goldens(synth):
    """The reference's own provider functions executed here: tokenize_mesh (naive and meto paths), detokenize_mesh (naive path),
    collate_fn on un-truncated and on all-truncated batches (a mixed batch makes the reference's np.stack raise)."""
    from core.provider import tokenize_mesh, detokenize_mesh, collate_fn
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import meshes
    opt = synth.tiny_options()
    out = {}

    class RefEnc:   # meto.Engine.encode surface over the compiled reference tokenizer (meto/meto/__init__.py:40-45)
        def __init__(self, bins):
            import _meto
            self.impl = _meto.Engine_LR_ABSCO(bins, False)

        def encode(self, vertices, faces):
            t, o, f = self.impl.encode(vertices, faces)
            return np.asarray(t), np.asarray(o), np.asarray(f)

    for name in ('cube', 'torus', 'icosphere', 'random_soup'):
        v, f = meshes.all_meshes()[name]
        v = v.astype(np.float64)
        out[f'tok_naive_{name}'] = np.asarray(tokenize_mesh(v, f, 512, tokenizer=None))
        out[f'tok_meto_{name}'] = np.asarray(tokenize_mesh(v, f, 512, tokenizer=RefEnc(512)))
        dv, df = detokenize_mesh(out[f'tok_naive_{name}'], 512, tokenizer=None)
        out[f'detok_naive_v_{name}'] = np.asarray(dv, dtype=np.float64)
        out[f'detok_naive_f_{name}'] = np.asarray(df, dtype=np.int64)
    for tag, lens in (('plain', [40, 13, 27, 40]), ('trunc', [opt.max_seq_length + 5, opt.max_seq_length + 90])):
        batch = provider_items(np.random.RandomState(5), opt, lens)
        res = collate_fn(batch, opt)
        for k in ('conds', 'num_faces', 'num_tokens', 'azimuths', 'tokens', 'labels', 'masks'):
            out[f'collate_{tag}_{k}'] = res[k].numpy()
        out[f'collate_{tag}_lens'] = np.asarray(lens)
    np.savez_compressed(os.path.join(GOLD, 'provider.npz'), **out)
    print('[gen] wrote provider.npz', flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--only', default='all')
    args = ap.parse_args()
    os.makedirs(GOLD, exist_ok=True)
    synth = import_reference()
    torch.set_num_threads(os.cpu_count())
    if args.only in ('all', 'meta'):
        gen_meta(synth)
    if args.only in ('all', 'meto'):
        gen_meto_goldens()
    if args.only in ('all', 'meto_clers'):
        gen_meto_clers_goldens()
    if args.only in ('all', 'meto_live'):
        gen_meto_live_goldens()
    if args.only in ('all', 'dit'):
        gen_dit_goldens()
    if args.only in ('all', 'provider'):
        gen_provider_goldens(synth)
    if args.only in ('all', 'train'):
        gen_train_goldens(synth)
    if args.only in ('all', 'tiny'):
        opt = synth.tiny_options()
        gen_model_goldens(synth, 'tiny', opt, steps=160, num_faces=1000, sample_steps=64, tf_len=40)
    if args.only in ('all', 'arae'):
        from core.options import config_defaults
        opt = dataclasses.replace(config_defaults['ArAE'], generate_mode='greedy')
        gen_model_goldens(synth, 'arae', opt, steps=40, num_faces=1000)


if __name__ == '__main__':
    main()
