"""Golden vectors of the REFERENCE's GPU path, for the GPU tests that compare this repository's CUDA path against it.

TEST INFRASTRUCTURE.  Executes the reference's own modules (copied by ``make -C oracle refpy`` into the git-ignored oracle/_ref,
run through oracle/ref_runner.py: ``model.half()``, ``torch.autocast('cuda', fp16)``, the installed flash-attn) on a CUDA device and
writes small ``.npz`` files; copy them to tests/golden/ (committed):

    python oracle/gen_golden_gpu.py [--out DIR] [--only lmm|dit|dropin]

  ref_gpu_lmm.npz    ArAE preset, synthetic weights (seed 0), point cloud 0: the reference's 600-token greedy stream; its fp16 logits
                     in full at 48 seeded positions and, at every position, the 8 best under the generation constraint (ids, values);
                     the forward-hook dtype ledger                                       -> tests/test_gpu_reference.py
  ref_gpu_dit.npz    DiT preset (24 layers), synthetic weights (seed 1): one guided-batch forward and an 8-step guided DDIM loop,
                     every DIT_STRIDE-th element of each output, their mean |x|, the dtype ledger  -> tests/test_gpu_dit.py
  dropin_infer.npz   the reference's unmodified infer.py run against this repository's core/ + meto/: the point cloud it sampled
                     and the tokens it wrote                                             -> tests/test_gpu_dropin.py
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
from dataclasses import replace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)

from oracle import ref_runner as rr  # noqa: E402

LMM_T, LMM_TOP, LMM_ROWS = 600, 8, 48
DIT_STRIDE, DIT_LOOP_STEPS = 17, 8


def _ledger_hooks(model, key_fn, ledger):
    def hook(name):
        def fn(mod, inp, out):
            i = inp[0] if isinstance(inp, tuple) and len(inp) else inp
            o = out[0] if isinstance(out, tuple) else out
            if torch.is_tensor(i) and torch.is_tensor(o):
                ledger.setdefault(key_fn(mod, name), set()).add(f'{str(i.dtype)[6:]}->{str(o.dtype)[6:]}')
        return fn
    return [m.register_forward_hook(hook(n)) for n, m in model.named_modules() if len(list(m.children())) == 0]


def gen_lmm(out_dir, dev, cfgs):
    from edgerunner_b200 import synth
    opt = replace(cfgs['ArAE'], generate_mode='greedy')
    sd = synth.synth_state_dict(opt, seed=0, eos_logit=-30.0)
    cond = synth.synth_point_cloud(0, opt.point_num).to(dev)
    model = rr.build_model(opt, sd, dev, half=True)
    del sd
    V = model.vocab_size
    ac = lambda: torch.autocast('cuda', dtype=torch.float16)  # noqa: E731

    ledger, phase = {}, ['prefill']

    def key(mod, name):
        last = name.split('.')[-1]
        return str((phase[0], type(mod).__name__, name if last.isdigit() else last))
    hs = _ledger_hooks(model, key, ledger)
    with torch.no_grad(), ac():
        emb = rr.prefix_embeds(model, cond, 4000)
        embeds_dtype = str(emb.dtype)
        rr.hf_sample(model.mesh_decoder, emb, opt.eos_token_id, 3, rr.fsm_fn(V, opt.eos_token_id), on_step=lambda n: phase.__setitem__(0, 'decode'))
    for h in hs:
        h.remove()

    rec = []
    with torch.no_grad(), ac():
        emb = rr.prefix_embeds(model, cond, 4000)
        tokens, _ = rr.hf_sample(model.mesh_decoder, emb, opt.eos_token_id, LMM_T, rr.fsm_fn(V, opt.eos_token_id), record_logits=rec)
    logits = torch.stack(rec)                                       # [T, V]: fp16 values
    assert len(tokens) == LMM_T, len(tokens)
    # the best LMM_TOP logits among the ids the generation constraint allows at each step (replayed on the stream)
    fsm = rr.fsm_fn(V, opt.eos_token_id)
    masked = torch.full_like(logits, -float('inf'))
    for t in range(LMM_T):
        allowed = fsm(0, torch.as_tensor(tokens[:t]))
        masked[t, allowed] = logits[t, allowed]
    top_vals, top_ids = torch.topk(masked, LMM_TOP, dim=1)
    assert torch.equal(top_vals[:, 0], masked.gather(1, torch.as_tensor(tokens)[:, None])[:, 0])      # greedy took the best allowed id
    rows = np.sort(np.random.RandomState(0).choice(LMM_T, LMM_ROWS, replace=False))
    np.savez_compressed(os.path.join(out_dir, 'ref_gpu_lmm.npz'), tokens=tokens.astype(np.int16), top_ids=top_ids.numpy().astype(np.int16),
                        top_vals=top_vals.numpy().astype(np.float16), rows=rows.astype(np.int16), row_logits=logits[rows].numpy().astype(np.float16),
                        ledger=json.dumps({k: sorted(v) for k, v in sorted(ledger.items())}), inputs_embeds_dtype=embeds_dtype)
    print('[gen] wrote ref_gpu_lmm.npz', flush=True)


def gen_dit(out_dir, dev):
    from core.transformer.dit import DiT                        # the reference's module
    from oracle import dit_oracle as do
    cfg = dict(hidden_dim=1024, num_heads=16, latent_size=2048, latent_dim=64, num_layers=24)
    M, B = 257, 2
    sd = do.synth_dit_state(**cfg, seed=1)
    ref = DiT(**cfg, gradient_checkpointing=False).eval()
    ref.load_state_dict(sd, strict=True)
    ref = ref.half().to(dev)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(B, cfg['latent_size'], cfg['latent_dim'], generator=g).to(dev)
    c = torch.randn(B, M, cfg['hidden_dim'], generator=g).to(dev)
    t = torch.tensor([991.0, 501.0]).to(dev)
    lat0 = torch.randn(1, cfg['latent_size'], cfg['latent_dim'], generator=g).to(dev)
    ac = lambda: torch.autocast('cuda', dtype=torch.float16)  # noqa: E731

    ledger = {}
    hs = _ledger_hooks(ref, lambda mod, name: f'{type(mod).__name__}:{name.split(".")[-1]}', ledger)
    with torch.no_grad(), ac():
        y = ref(x, c, t)
    for h in hs:
        h.remove()

    # MDiT.run's loop body with the reference module as the denoiser: guidance 7.5 + the restated diffusers DDIM step
    ts, coef = do.ddim_tables(DIT_LOOP_STEPS)
    lat, cond = lat0.clone(), c[:1]
    cc = torch.cat([torch.zeros_like(cond), cond], dim=0)
    with torch.no_grad(), ac():
        for i, tt in enumerate(ts.tolist()):
            pred = ref(torch.cat([lat] * 2, dim=0), cc, torch.tensor([tt] * 2, device=dev, dtype=lat.dtype))
            u, cnd = pred.chunk(2)
            lat = do.ddim_step((u + 7.5 * (cnd - u)).float(), lat, coef[i], 'v_prediction', ledger=True)
    yf, lf = y.float().cpu().reshape(-1), lat.float().cpu().reshape(-1)
    np.savez_compressed(os.path.join(out_dir, 'ref_gpu_dit.npz'), out_dtype=str(y.dtype), out_sample=yf[::DIT_STRIDE].numpy().astype(np.float16),
                        out_abs_mean=float(yf.abs().mean()), loop_sample=lf[::DIT_STRIDE].numpy(), loop_abs_mean=float(lf.abs().mean()),
                        stride=DIT_STRIDE, loop_steps=DIT_LOOP_STEPS, ledger=json.dumps({k: sorted(v) for k, v in sorted(ledger.items())}))
    print('[gen] wrote ref_gpu_dit.npz', flush=True)


def gen_dropin(out_dir, cfgs):
    """infer.py as a user runs it, on a unit cube with a small synthetic checkpoint; its PYTHONPATH puts this repository's core/ + meto/
    first (tests/stubs provides the import-time and I/O calls of kiui / trimesh)."""
    from safetensors.torch import save_file
    from edgerunner_b200 import synth
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    from test_gpu_dropin import DIMS, _write_obj
    infer = os.path.join(HERE, '_ref', 'drop_in', 'infer.py')
    opt = replace(cfgs['ArAE'], hidden_dim=768, num_heads=8, num_layers=2, point_hidden_dim=128, point_num_heads=2,
                  point_latent_size=64, point_latent_dim=16, point_num=256, num_cond_tokens=65, max_seq_length=512, generate_mode='greedy')
    with tempfile.TemporaryDirectory() as tmp:
        sd = synth.synth_state_dict(opt, seed=9, eos_logit=-30.0)
        ckpt = os.path.join(tmp, 'synthetic.safetensors')
        save_file({k: v.contiguous() for k, v in sd.items()}, ckpt)
        obj = os.path.join(tmp, 'cube.obj')
        _write_obj(obj)
        ws = os.path.join(tmp, 'ws')
        env = dict(os.environ, PYTHONPATH=os.pathsep.join([REPO, os.path.join(REPO, 'tests', 'stubs')]))
        cmd = [sys.executable, infer, 'ArAE', '--test_path', obj, '--workspace', ws, '--resume', ckpt, '--test_num_face', '1000',
               '--test_max_seq_length', '96', '--test_repeat', '1'] + DIMS
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=tmp)
        assert out.returncode == 0, (out.stdout[-1500:], out.stderr[-3000:])
        assert 'Loaded checkpoint' in out.stdout
        ply, npy, pc = os.path.join(ws, 'cube_0_1000f.ply'), os.path.join(ws, 'cube_0_1000f_tokens.npy'), os.path.join(ws, 'cube_pc.obj')
        head = open(ply).read(200)
        assert head.startswith('ply') and 'element face' in head
        toks = np.load(npy)
        pts = np.asarray([[float(x) for x in l.split()[1:4]] for l in open(pc) if l.startswith('v ')], dtype=np.float64)
    assert pts.shape == (256, 3) and len(toks) == 96
    np.savez_compressed(os.path.join(out_dir, 'dropin_infer.npz'), points=pts.astype(np.float32), tokens=toks.astype(np.int16))
    print('[gen] wrote dropin_infer.npz', flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(REPO, 'tests', 'golden'))
    ap.add_argument('--only', default='all', choices=['all', 'lmm', 'dit', 'dropin'])
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device('cuda:0')
    use_flash = rr.flash_usable(dev)
    print('[gen] flash-attn used:', use_flash, '| device:', torch.cuda.get_device_name(0), flush=True)
    _, cfgs = rr.setup(mask_flash=not use_flash)
    if args.only in ('all', 'dropin'):
        gen_dropin(args.out, cfgs)
    if args.only in ('all', 'lmm'):
        gen_lmm(args.out, dev, cfgs)
    if args.only in ('all', 'dit'):
        gen_dit(args.out, dev)


if __name__ == '__main__':
    main()
