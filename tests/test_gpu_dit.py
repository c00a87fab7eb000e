"""GPU parity of the DiT denoiser path (SURVEY.md §8 f3): the CUDA engine behind the C ABI (`er_dit_*`) against
  * the oracle (oracle/dit_oracle.py, ledger mode = fp16 rounding points of .half() + autocast) at a tiny and at the preset's layer shape,
  * the REFERENCE's own DiT module on a B200 (.half() + autocast + flash-attn, recorded in tests/golden) at the full 24-layer preset,
  * for the sampling loop: the oracle's loop (reference MDiT.run + restated diffusers DDIM step), graph replay vs direct launches bit for bit,
  * MDiT.run -> LMM.generate(point_latent) plumbing (infer_dit.py:104-113).
Tolerances are on fp16 outputs of O(1) magnitude: two correct fp16 pipelines differ by accumulation order inside GEMMs / softmax."""
import dataclasses
import json
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, 'oracle'))


def _engine(cfg, M, sd_full, cond_dim):
    from edgerunner_b200.dit_engine import DiTEngine
    eng = DiTEngine(torch.device('cuda:0'), cfg['hidden_dim'], cfg['num_heads'], cfg['num_layers'], cfg['latent_size'], cfg['latent_dim'], M, cond_dim)
    eng.load_state_dict(sd_full)
    return eng


def _case(cfg, M, B, cond_dim=32, seed=0):
    from dit_oracle import DitOracle, synth_dit_state
    sd = synth_dit_state(**cfg, cond_dim=cond_dim, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, cfg['latent_size'], cfg['latent_dim'], generator=g).cuda()
    c = torch.randn(B, M, cfg['hidden_dim'], generator=g).cuda()
    t = torch.tensor([991.0, 3.0, 500.0, 41.0, 77.0][:B]).cuda()
    return sd, x, c, t, DitOracle(sd, cfg['num_heads'], mode='ledger', device='cuda'), _engine(cfg, M, sd, cond_dim)


def test_dit_forward_matches_oracle_tiny_ragged():
    """latent_size 40 / 9 condition tokens (tails of every tile), 3 samples with different timesteps, head_dim 64."""
    cfg = dict(hidden_dim=128, num_heads=2, latent_size=40, latent_dim=16, num_layers=2)
    sd, x, c, t, orc, eng = _case(cfg, 9, 3)
    y = eng.forward(x, c, t)
    assert y.dtype == torch.float16 and y.shape == x.shape
    ref = orc.forward(x, c, t)
    d = (y.float() - ref).abs()
    print('tiny: max', float(d.max()), 'mean', float(d.mean()), 'ref mean abs', float(ref.abs().mean()))
    assert float(ref.abs().mean()) > 0.1 and float(d.max()) <= 2e-2 and float(d.mean()) <= 1.5e-3
    # the adaptor: norm_cond(proj_cond(h))
    h = torch.randn(3, 9, 32, device='cuda').half()
    a = eng.cond(h)
    ra = orc.cond_adaptor(h.float())
    assert a.dtype == torch.float32 and float((a - ra).abs().max()) <= 5e-3
    # repeatable bit for bit; GEGLU / gated residuals fused into the GEMM epilogues (default) == the separate kernels, bit for bit
    assert torch.equal(y, eng.forward(x, c, t))
    eng.debug_set('fuse', 0)
    assert torch.equal(y, eng.forward(x, c, t))
    eng.debug_set('fuse', 1)


def test_dit_forward_head_dim_96_generic_width():
    """hidden 192 = 2 heads of 96: the D = 96 attention kernel (non-causal, ragged), the generic-width LayerNorm kernel."""
    cfg = dict(hidden_dim=192, num_heads=2, latent_size=72, latent_dim=8, num_layers=2)
    sd, x, c, t, orc, eng = _case(cfg, 5, 2, seed=2)
    y = eng.forward(x, c, t).float()
    ref = orc.forward(x, c, t)
    d = (y - ref).abs()
    print('d96: max', float(d.max()), 'mean', float(d.mean()))
    assert float(ref.abs().mean()) > 0.1 and float(d.max()) <= 2e-2 and float(d.mean()) <= 1.5e-3
    eng.debug_set('fuse', 0)
    assert torch.equal(y, eng.forward(x, c, t).float())


def test_dit_forward_matches_oracle_preset_shape():
    """the preset's layer shape (1024 wide, 16 heads, 2048 latents, 257 CLIP tokens), 3 layers, batch 2."""
    cfg = dict(hidden_dim=1024, num_heads=16, latent_size=2048, latent_dim=64, num_layers=3)
    sd, x, c, t, orc, eng = _case(cfg, 257, 2, cond_dim=1280)
    y = eng.forward(x, c, t).float()
    ref = orc.forward(x, c, t)
    d = (y - ref).abs()
    print('preset shape: max', float(d.max()), 'mean', float(d.mean()), 'ref mean abs', float(ref.abs().mean()))
    assert float(ref.abs().mean()) > 0.1 and float(d.max()) <= 3e-2 and float(d.mean()) <= 2e-3


@pytest.mark.parametrize('ptype', ['v_prediction', 'epsilon'])
def test_sampling_loop_matches_oracle(ptype):
    """6 guided DDIM steps on the device (CUDA graph per step) vs the oracle's loop; graph replay == direct launches bit for bit;
    a second run with another step count / init step reuses the engine."""
    from dit_oracle import ddim_tables
    cfg = dict(hidden_dim=128, num_heads=2, latent_size=40, latent_dim=16, num_layers=2)
    sd, x, c, t, orc, eng = _case(cfg, 9, 2, seed=4)
    ts, coef = ddim_tables(6)
    lat0 = x.clone()
    ref = orc.sample_loop(c, lat0, ts.tolist(), coef, 7.5, ptype)
    out = eng.run(c, lat0.clone(), ts.astype(np.float32), coef.numpy(), 7.5, True, ptype)
    d = (out - ref).abs()
    print(ptype, 'loop: max', float(d.max()), 'mean', float(d.mean()), 'latent mean abs', float(ref.abs().mean()))
    # guidance multiplies the fp16 difference of two predictions by 7.5 every step and the epsilon form divides by sqrt(alpha_t) = 0.07 at
    # t = 991: the tolerance is relative to the latents' magnitude (a random network drives them to |x| ~ 4 (v) / ~ 18 (epsilon))
    scale = max(1.0, float(ref.abs().mean()))
    assert torch.isfinite(out).all() and float(d.max()) <= 1.5e-2 * scale and float(d.mean()) <= 2e-3 * scale
    n0 = eng.kernel_launches()
    again = eng.run(c, lat0.clone(), ts.astype(np.float32), coef.numpy(), 7.5, True, ptype)
    assert torch.equal(out, again)
    assert eng.kernel_launches() - n0 >= 6 * (6 + 10 * cfg['num_layers'])
    eng.debug_set('graph', 0)
    direct = eng.run(c, lat0.clone(), ts.astype(np.float32), coef.numpy(), 7.5, True, ptype)
    assert torch.equal(out, direct)
    eng.debug_set('graph', 1)
    # the zero-condition half's cross-attention replaced by its closed form (default) == computing it in full, bit for bit
    eng.debug_set('uncond_shortcut', 0)
    assert torch.equal(out, eng.run(c, lat0.clone(), ts.astype(np.float32), coef.numpy(), 7.5, True, ptype))
    eng.debug_set('uncond_shortcut', 1)
    # strength path: start in the middle of a longer schedule; unguided variant runs too
    ts2, coef2 = ddim_tables(10)
    part = eng.run(c, lat0.clone(), ts2[4:].astype(np.float32), coef2[4:].numpy(), 3.0, True, ptype)
    ref2 = orc.sample_loop(c, lat0, ts2[4:].tolist(), coef2[4:], 3.0, ptype)
    assert float((part - ref2).abs().max()) <= 1.5e-2 * max(1.0, float(ref2.abs().mean()))
    ung = eng.run(c, lat0.clone(), ts.astype(np.float32), coef.numpy(), 1.0, False, ptype)
    assert torch.isfinite(ung).all() and not torch.equal(ung, out)


def test_reference_dit_module_on_gpu_against_engine(golden_dir):
    """The reference's DiT (24 layers, preset size) executed on a B200 as infer_dit.py runs it (.half() + autocast + flash-attn), vs the
    engine: forward and an 8-step guided loop.  The reference's outputs are recorded in ref_gpu_dit.npz (oracle/gen_golden_gpu.py):
    every 17th element of each, their mean |x| and its dtype ledger; inputs and weights are regenerated from the same seeds."""
    from dit_oracle import DitOracle, ddim_tables, synth_dit_state
    g = np.load(os.path.join(golden_dir, 'ref_gpu_dit.npz'))
    cfg = dict(hidden_dim=1024, num_heads=16, latent_size=2048, latent_dim=64, num_layers=24)
    M, B, S, stride = 257, 2, int(g['loop_steps']), int(g['stride'])
    sd = synth_dit_state(**cfg, seed=1)
    gen = torch.Generator().manual_seed(2)
    x = torch.randn(B, cfg['latent_size'], cfg['latent_dim'], generator=gen).cuda()
    c = torch.randn(B, M, cfg['hidden_dim'], generator=gen).cuda()
    t = torch.tensor([991.0, 501.0]).cuda()
    lat0 = torch.randn(1, cfg['latent_size'], cfg['latent_dim'], generator=gen).cuda()
    full = {'dit.' + k: v for k, v in sd.items()}
    C = cfg['hidden_dim']
    full.update({'proj_cond.weight': torch.zeros(C, 1280), 'proj_cond.bias': torch.zeros(C), 'norm_cond.weight': torch.ones(C), 'norm_cond.bias': torch.zeros(C)})
    eng = _engine(cfg, M, full, 1280)
    y_ref = torch.as_tensor(g['out_sample']).float()
    y_orc = DitOracle(sd, cfg['num_heads'], mode='ledger', device='cuda').forward(x, c, t).float().cpu().reshape(-1)[::stride]
    y = eng.forward(x, c, t).float().cpu().reshape(-1)[::stride]
    ts, coef = ddim_tables(S)
    lat = eng.run(c[:1], lat0.clone(), ts.astype(np.float32), coef.numpy(), 7.5, True, 'v_prediction').float().cpu().reshape(-1)[::stride]
    lat_ref, lat_abs_mean = torch.as_tensor(g['loop_sample']), float(g['loop_abs_mean'])
    d = {'engine_vs_ref': {'max': float((y - y_ref).abs().max()), 'mean': float((y - y_ref).abs().mean())},
         'oracle_vs_ref': {'max': float((y_orc - y_ref).abs().max()), 'mean': float((y_orc - y_ref).abs().mean())},
         'loop_engine_vs_ref': {'steps': S, 'max': float((lat - lat_ref).abs().max()), 'mean': float((lat - lat_ref).abs().mean()), 'lat_abs_mean': lat_abs_mean}}
    print('reference DiT on GPU vs engine:', json.dumps(d))
    assert str(g['out_dtype']) == 'torch.float16'
    led = json.loads(str(g['ledger']))
    for k, v in led.items():                         # the ledger the kernels implement: Linear -> fp16, LayerNorm -> fp32
        if k.startswith('Linear:'):
            assert all(x.endswith('->float16') for x in v), (k, v)
        if k.startswith('LayerNorm:'):
            assert all(x.endswith('->float32') for x in v), (k, v)
    assert 'float16->float32' in led['LayerNorm:norm1'] and 'float32->float32' in led['LayerNorm:norm1']      # layer 0 sees fp16, later layers the fp32 stream
    assert float(g['out_abs_mean']) > 0.1
    assert d['engine_vs_ref']['max'] <= 4e-2 and d['engine_vs_ref']['mean'] <= 3e-3, d['engine_vs_ref']
    assert d['oracle_vs_ref']['max'] <= 4e-2 and d['oracle_vs_ref']['mean'] <= 3e-3, d['oracle_vs_ref']
    lp = d['loop_engine_vs_ref']
    assert lp['max'] <= 3e-2 * max(1.0, lp['lat_abs_mean']) and lp['mean'] <= 3e-3 * max(1.0, lp['lat_abs_mean']), lp


def test_mdit_run_feeds_lmm_generate():
    """infer_dit.py:104-113 plumbing at a small size: MDiT.run(image) -> latents [1, N, Dl] fp32 -> LMM.generate in point_latent mode."""
    from core.options import config_defaults
    from core.models_dit import MDiT
    from core.models import LMM
    from edgerunner_b200 import synth
    from dit_oracle import DitOracle
    opt = dataclasses.replace(synth.tiny_options(), cond_mode='point_latent', dit_hidden_dim=128, dit_num_heads=2, dit_num_layers=2, noise_scheduler_predtype='v_prediction')
    tiny_clip = dict(hidden_size=32, intermediate_size=64, num_hidden_layers=2, num_attention_heads=2, image_size=28, patch_size=14, hidden_act='gelu')
    torch.manual_seed(0)
    mdit = MDiT(opt, image_encoder_config=tiny_clip).half().eval().cuda()
    img = torch.rand(1, 3, 64, 64, device='cuda')
    torch.manual_seed(7)
    lat = mdit.run(img, num_inference_steps=5, guidance_scale=4.0)
    assert lat.shape == (1, opt.point_latent_size, opt.point_latent_dim) and lat.dtype == torch.float32 and torch.isfinite(lat).all()
    # the same through the oracle: same cond (from the engine's adaptor check below), same initial noise
    cond = mdit.get_cond(img)
    orc = DitOracle({k: v for k, v in mdit.state_dict().items() if k.startswith(('dit.', 'proj_cond', 'norm_cond'))}, opt.dit_num_heads, 'ledger', 'cuda')
    with torch.no_grad():
        size = mdit.image_encoder.config.image_size
        h = mdit.image_encoder(torch.nn.functional.interpolate(mdit.normalize_image(img), (size, size), mode='bilinear', align_corners=False).half()).last_hidden_state
    assert float((orc.cond_adaptor(h.float()) - cond).abs().max()) <= 5e-3
    torch.manual_seed(7)
    noise = torch.randn(1, opt.point_latent_size, opt.point_latent_dim, device='cuda', dtype=torch.float32)
    mdit.scheduler.set_timesteps(5)
    ts = mdit.scheduler.timesteps
    ref = orc.sample_loop(cond, noise, ts.tolist(), mdit.scheduler.step_coefficients(ts), 4.0, 'v_prediction')
    assert float((lat - ref).abs().max()) <= 1.5e-2 * max(1.0, float(ref.abs().mean()))
    # num_repeat: the condition is repeated, every copy gets its own noise
    torch.manual_seed(9)
    rep = mdit.run(img, num_inference_steps=3, guidance_scale=4.0, num_repeat=2)
    assert rep.shape == (2, opt.point_latent_size, opt.point_latent_dim) and not torch.equal(rep[0], rep[1]) and torch.isfinite(rep).all()
    # strength path of run()
    torch.manual_seed(8)
    lat2 = mdit.run(img, num_inference_steps=6, guidance_scale=4.0, latents=lat, strength=0.5)
    assert lat2.shape == lat.shape and torch.isfinite(lat2).all()
    # then run lmm (infer_dit.py:111-113)
    from core.utils import get_tokenizer
    lopt = synth.tiny_options(cond_mode='point_latent')
    lmm = LMM(lopt)
    lmm.load_state_dict(synth.synth_state_dict(lopt, seed=1, eos_logit=-30.0), strict=True)
    lmm = lmm.half().eval().cuda()
    tok, _ = get_tokenizer(lopt)
    meshes, tokens = lmm.generate(lat, num_faces=1000, max_new_tokens=64, tokenizer=tok, clean=True)
    assert len(tokens) == 1 and len(tokens[0]) == 64 and len(meshes) == 1


def test_dit_abi_error_behaviour():
    """strict weight loading and state checks of the er_dit_* entry points (the reference raises on shape mismatches in load_state_dict)."""
    from edgerunner_b200 import _lib
    from edgerunner_b200.dit_engine import DiTEngine
    from dit_oracle import synth_dit_state
    cfg = dict(hidden_dim=128, num_heads=2, latent_size=40, latent_dim=16, num_layers=1)
    sd = synth_dit_state(**cfg, cond_dim=32, seed=0)
    with pytest.raises(_lib.ErError):                                   # head_dim 32 is not a kernel shape
        DiTEngine(torch.device('cuda:0'), 64, 2, 1, 40, 16, 9, 32)
    eng = DiTEngine(torch.device('cuda:0'), 128, 2, 1, 40, 16, 9, 32)
    x, c, t = torch.zeros(1, 40, 16).cuda(), torch.zeros(1, 9, 128).cuda(), torch.zeros(1).cuda()
    with pytest.raises(_lib.ErError):                                   # not finalized
        eng.forward(x, c, t)
    with pytest.raises(_lib.ErError):                                   # a tensor of the schema is missing
        eng.load_state_dict({k: v for k, v in sd.items() if k != 'dit.proj_out.bias'})
    with pytest.raises(_lib.ErError):                                   # wrong element count
        eng.load_state_dict({**sd, 'dit.proj_in.bias': torch.zeros(7)})
    with pytest.raises(_lib.ErError):                                   # unknown dit.* key
        eng.load_state_dict({**sd, 'dit.layers.0.attn3.weight': torch.zeros(4)})
    eng.load_state_dict({**sd, 'image_encoder.foo': torch.zeros(3), 'point_encoder.bar': torch.zeros(3)})     # not the engine's keys: ignored
    assert torch.isfinite(eng.forward(x, c, t).float()).all()
    with pytest.raises(_lib.ErError):
        eng.debug_set('no_such_switch', 1)
