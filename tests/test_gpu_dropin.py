"""The drop-in claim, executed (VERDICT r1 item 7): the reference's UNMODIFIED `infer.py` runs against THIS repository's `core/` + `meto/`
packages on a synthetic .obj with a synthetic checkpoint, writes the .ply and the _tokens.npy it promises, and the tokens equal what
`LMM.generate` returns in-process for the same sampled point cloud (that run is recorded in tests/golden/dropin_infer.npz).  The
image-conditioned script infer_dit.py runs from the git-ignored oracle/_ref/drop_in/ (`make -C oracle refpy`) when that copy is present.
`kiui` / `trimesh` are absent from the image: tests/stubs/ provides the few import-time and I/O calls the scripts make (seeded surface
sampling, .obj load, exports); no arithmetic of the path lives there."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DIMS = ['--generate_mode', 'greedy', '--hidden_dim', '768', '--num_heads', '8', '--num_layers', '2', '--point_hidden_dim', '128', '--point_num_heads', '2',
        '--point_latent_size', '64', '--point_latent_dim', '16', '--point_num', '256', '--num_cond_tokens', '65', '--max_seq_length', '512']


def _write_obj(path):
    """a unit cube, 12 triangles"""
    v = [(x, y, z) for x in (0, 1) for y in (0, 1) for z in (0, 1)]
    f = [(0, 1, 3), (0, 3, 2), (4, 6, 7), (4, 7, 5), (0, 4, 5), (0, 5, 1), (2, 3, 7), (2, 7, 6), (0, 2, 6), (0, 6, 4), (1, 5, 7), (1, 7, 3)]
    with open(path, 'w') as fh:
        for p in v:
            fh.write('v %g %g %g\n' % p)
        for t in f:
            fh.write('f %d %d %d\n' % tuple(i + 1 for i in t))


def test_reference_infer_py_runs_unmodified(golden_dir):
    """What the unmodified infer.py wrote when run against this repository (the point cloud it sampled from a unit cube, the tokens of
    its .npy; recorded in dropin_infer.npz by oracle/gen_golden_gpu.py, which also checks the .ply it writes) equals what LMM.generate
    returns in-process for the same cloud and synthetic checkpoint."""
    from dataclasses import replace
    from core.models import LMM
    from core.options import config_defaults
    from core.utils import get_tokenizer
    from edgerunner_b200 import synth
    g = np.load(os.path.join(golden_dir, 'dropin_infer.npz'))
    toks_file, pts = g['tokens'].astype(np.int64), g['points']
    assert len(toks_file) == 96 and toks_file[0] == 2             # BOM (5) - 3; no EOS with the synthetic checkpoint
    assert pts.shape == (256, 3)
    opt = replace(config_defaults['ArAE'], hidden_dim=768, num_heads=8, num_layers=2, point_hidden_dim=128, point_num_heads=2,
                  point_latent_size=64, point_latent_dim=16, point_num=256, num_cond_tokens=65, max_seq_length=512, generate_mode='greedy')
    sd = synth.synth_state_dict(opt, seed=9, eos_logit=-30.0)
    model = LMM(opt)
    model.load_state_dict(sd, strict=False)
    model = model.half().eval().to('cuda')
    tokenizer, _ = get_tokenizer(opt)
    cond = torch.from_numpy(pts).unsqueeze(0).float().to('cuda')
    with torch.no_grad(), torch.autocast(device_type='cuda', dtype=torch.float16):
        meshes, tokens = model.generate(cond, num_faces=1000, max_new_tokens=96, tokenizer=tokenizer, clean=True)
    np.testing.assert_array_equal(tokens[0] - 3, toks_file)
    assert len(meshes[0].faces) > 0


INFER_DIT = os.path.join(REPO, 'oracle', '_ref', 'drop_in', 'infer_dit.py')


@pytest.mark.skipif(not os.path.exists(INFER_DIT), reason='oracle/_ref/drop_in/infer_dit.py missing: run `make -C oracle refpy` in the build container')
def test_reference_infer_dit_py_runs_unmodified(tmp_path):
    """The image-conditioned script (infer_dit.py:34-144), unmodified, against this repository's core/ (LMM, MDiT, DiT) + meto/: RGBA image ->
    CLIP tower (random ViT-H/14: no network) -> MDiT.run (100 guided DDIM steps on the device) -> LMM.generate(point_latent) -> .obj + tokens.
    Small LMM / DiT dimensions through the script's own tyro flags; rembg / kiui image I/O are tests/stubs."""
    from PIL import Image
    rng = np.random.RandomState(0)
    img = np.zeros((96, 96, 4), dtype=np.uint8)
    img[24:72, 30:66, :3] = rng.randint(0, 255, (48, 36, 3))
    img[24:72, 30:66, 3] = 255
    path = str(tmp_path / 'blob.png')
    Image.fromarray(img, 'RGBA').save(path)
    ws = str(tmp_path / 'ws')
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([REPO, os.path.join(REPO, 'tests', 'stubs')]))
    cmd = [sys.executable, INFER_DIT, 'DiT', '--test_path', path, '--workspace', ws, '--test_num_face', '1000', '--test_max_seq_length', '64',
           '--test_repeat', '1', '--dit_hidden_dim', '128', '--dit_num_heads', '2', '--dit_num_layers', '2'] + DIMS
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=str(tmp_path))
    assert out.returncode == 0, (out.stdout[-1500:], out.stderr[-3000:])
    obj, npy = os.path.join(ws, 'blob_0_1000f.obj'), os.path.join(ws, 'blob_0_1000f_tokens.npy')
    assert os.path.exists(obj) and os.path.exists(npy) and os.path.exists(os.path.join(ws, 'blob.jpg')), os.listdir(ws)
    toks = np.load(npy)
    assert 1 <= len(toks) <= 64 and toks[0] == 2                   # BOM (5) - 3 first; a randomly initialised LMM may emit EOS before 64 tokens
    assert open(obj).read(2) == 'v '
