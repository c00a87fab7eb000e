"""meto detokenizer: native C-ABI implementation and the C oracle against the compiled-reference goldens (CPU)."""

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def oracle_lib():
    path = os.path.join(REPO, 'oracle', 'libmeto_oracle.so')
    if not os.path.exists(path):
        subprocess.check_call(['make', '-C', os.path.join(REPO, 'oracle'), 'oracle'])
    return C.CDLL(path)


def oracle_decode(lib, bins, tok):
    tok = np.ascontiguousarray(tok, dtype=np.int32)
    n = len(tok)
    cap = n // 4 + 3
    v = np.empty((3 * cap, 3), np.float32); f = np.empty((cap, 3), np.int32); t = np.empty(cap, np.int32)
    nv, nf, nt = C.c_int64(), C.c_int64(), C.c_int64()
    P = lambda a, ty: a.ctypes.data_as(C.POINTER(ty))
    lib.meto_oracle_decode(C.c_int(bins), P(tok, C.c_int32), C.c_int64(n), P(v, C.c_float), P(f, C.c_int32), P(t, C.c_int32),
                           C.byref(nv), C.byref(nf), C.byref(nt))
    return v[:nv.value].astype(np.float64), f[:nf.value], t[:nt.value]


def cases(golden_dir):
    g = np.load(os.path.join(golden_dir, 'meto.npz'))
    for key in g['names']:
        key = str(key)
        yield key, int(key.rsplit('_', 1)[1]), g[key + '_tokens'], g[key + '_dv'], g[key + '_df'], g[key + '_dt']
    for i in range(int(g['n_streams'])):
        yield f'stream{i}', 512, g[f'stream{i}_tokens'], g[f'stream{i}_dv'], g[f'stream{i}_df'], g[f'stream{i}_dt']


def test_oracle_matches_reference(golden_dir, oracle_lib):
    n = 0
    for name, bins, tok, dv, df, dt in cases(golden_dir):
        v, f, t = oracle_decode(oracle_lib, bins, tok)
        np.testing.assert_array_equal(v, dv.reshape(-1, 3), err_msg=name)      # bit-exact (float32 values)
        np.testing.assert_array_equal(f, df.reshape(-1, 3), err_msg=name)
        np.testing.assert_array_equal(t, dt, err_msg=name)
        n += 1
    assert n >= 30


def test_oracle_lr_matches_reference(golden_dir, oracle_lib):
    """The LR restatement (oracle/meto_oracle.c::meto_oracle_decode_lr) against the compiled reference's Engine_LR.decode."""
    g = np.load(os.path.join(golden_dir, 'meto.npz'))
    keys = [(str(k) + '_tokens', str(k) + '_dv', str(k) + '_df', str(k) + '_dt') for k in g['lr_names']]
    keys += [(f'lr_stream{i}_tokens', f'lr_stream{i}_dv', f'lr_stream{i}_df', f'lr_stream{i}_dt') for i in range(int(g['n_lr_streams']))]
    P = lambda a, ty: a.ctypes.data_as(C.POINTER(ty))
    for kt, kv, kf, ktt in keys:
        tok = np.ascontiguousarray(g[kt], dtype=np.int32)
        n = len(tok); cap = n // 4 + 3
        v = np.empty((3 * cap, 3), np.float32); f = np.empty((cap, 3), np.int32); t = np.empty(cap, np.int32)
        nv, nf, nt = C.c_int64(), C.c_int64(), C.c_int64()
        oracle_lib.meto_oracle_decode_lr(C.c_int(512), P(tok, C.c_int32), C.c_int64(n), P(v, C.c_float), P(f, C.c_int32), P(t, C.c_int32),
                                         C.byref(nv), C.byref(nf), C.byref(nt))
        np.testing.assert_array_equal(v[:nv.value].astype(np.float64), g[kv].reshape(-1, 3), err_msg=kt)
        np.testing.assert_array_equal(f[:nf.value], g[kf].reshape(-1, 3), err_msg=kt)
        np.testing.assert_array_equal(t[:nt.value], g[ktt], err_msg=kt)
    assert len(keys) >= 15


def test_native_matches_reference(golden_dir):
    from meto import Engine
    for name, bins, tok, dv, df, dt in cases(golden_dir):
        v, f, t = Engine(bins).decode(tok)
        assert v.dtype == np.float64
        np.testing.assert_array_equal(v, dv.reshape(-1, 3), err_msg=name)
        np.testing.assert_array_equal(f, df.reshape(-1, 3), err_msg=name)
        np.testing.assert_array_equal(t, dt, err_msg=name)


def test_cube_known_answer():
    """KAT recorded from the compiled reference in SURVEY.md §8c (cube scaled to +-0.95, bins 512)."""
    from meto import Engine
    tok = [2, 502, 15, 502, 502, 15, 15, 15, 15, 15, 0, 15, 15, 502, 0, 15, 502, 15, 0, 502, 502, 15, 0, 502, 15, 15, 1, 502, 502, 502,
           0, 502, 15, 502, 1, 15, 15, 502, 1, 15, 502, 502, 0, 15, 502, 15, 1, 502, 502, 15, 1, 502, 502, 502]
    v, f, t = Engine(512).decode(np.array(tok))   # _meto alphabet (already -3): 2 = BOM, coords +3
    assert v.shape == (14, 3) and f.shape == (12, 3)
    assert t.tolist() == [0, 0, 0, 0, 1, 0, 1, 1, 0, 1, 1, 2]
    assert v.max() == 0.951171875


def test_save_mesh_tail(golden_dir):
    """provider.save_mesh: EOS cut + detokenize (core/provider.py:39-66) on the tiny golden token stream."""
    from core.provider import save_mesh
    from edgerunner_b200 import synth
    from meto import Engine
    g = np.load(os.path.join(golden_dir, 'tiny.npz'))
    opt = synth.tiny_options()
    mesh = save_mesh(g['greedy_tokens'], opt, tokenizer=Engine(opt.discrete_bins), clean=False)
    np.testing.assert_array_equal(np.asarray(mesh.vertices), g['mesh_vertices'])
    np.testing.assert_array_equal(np.asarray(mesh.faces), g['mesh_faces'])


# ------------------------------------------------------------------ encode (training-data side) ------------------------------------------------------------------

def test_encode_matches_reference_goldens(golden_dir):
    """er_meto_encode vs token streams / face order / face types recorded from the compiled reference (bit-exact)."""
    import meshes
    from meto import Engine
    g = np.load(os.path.join(golden_dir, 'meto.npz'))
    fixtures = dict(meshes.all_meshes())
    fixtures.update(meshes.stress_meshes())
    n = 0
    for key in list(g['names']) + list(g['enc_names']):
        key = str(key)
        name, bins = key.rsplit('_', 1)
        v, f = fixtures[name]
        tok, order, ftype = Engine(int(bins)).encode(v, f)
        assert tok.dtype == np.int64
        np.testing.assert_array_equal(tok, g[key + '_tokens'], err_msg=key)
        np.testing.assert_array_equal(order, g[key + '_order'], err_msg=key)
        np.testing.assert_array_equal(ftype, g[key + '_ftype'], err_msg=key)
        n += 1
    assert n >= 100


def test_encode_live_against_compiled_reference(golden_dir):
    """Random jittered grids (meshes.random_grids) against the compiled reference's Engine_LR_ABSCO / Engine_LR on the same meshes,
    recorded in meto_live.npz (oracle/gen_golden.py --only meto_live): encode and decode, bit-exact."""
    import meshes
    from meto import Engine
    g = np.load(os.path.join(golden_dir, 'meto_live.npz'))
    ref = {k: np.split(g[k], np.cumsum(g['n_' + k])[:-1]) for k in ('tokens', 'order', 'ftype', 'dv', 'df', 'dt')}
    n = 0
    for it, v, f, bins in meshes.random_grids():
        for backend in ('LR_ABSCO', 'LR'):
            msg = f'{backend} iter {it}'
            assert int(g['bins'][n]) == bins, msg
            eng = Engine(bins, backend=backend)
            tok, order, ftype = eng.encode(v, f)
            np.testing.assert_array_equal(tok, ref['tokens'][n], err_msg=msg)
            np.testing.assert_array_equal(order, ref['order'][n], err_msg=msg)
            np.testing.assert_array_equal(ftype, ref['ftype'][n], err_msg=msg)
            mv, mf, mt = eng.decode(tok)
            np.testing.assert_array_equal(mv, ref['dv'][n].astype(np.float64), err_msg=msg)
            np.testing.assert_array_equal(mf, ref['df'][n], err_msg=msg)
            np.testing.assert_array_equal(mt, ref['dt'][n], err_msg=msg)
            n += 1
    assert n == len(g['bins']) == 80


def test_encode_decode_round_trip():
    """Size-independent properties: every face is emitted once; decode(encode(mesh)) reproduces each input face's quantised
    corner set, in emission order (the reference's own round-trip check, meto/tests/engine.py:120-150)."""
    import meshes
    from meto import Engine
    bins = 512
    for name, (v, f) in {**meshes.all_meshes(), 'icosphere4': meshes.icosphere(4)}.items():
        eng = Engine(bins)
        tok, order, ftype = eng.encode(v, f)
        assert sorted(order.tolist()) == list(range(len(f))), name
        assert len(ftype) == len(f)
        assert (tok == 2).sum() == (ftype == 2).sum(), name          # one BOM per strip end
        assert len(tok) == 4 * len(f) + 6 * (tok == 2).sum(), name   # 10 tokens for a strip's first face, 4 for the others
        dv, df, dt = eng.decode(tok)
        assert len(df) == len(f), name
        np.testing.assert_array_equal(dt, ftype, err_msg=name)
        q = np.minimum(((v.astype(np.float32) + 1) * bins / 2).astype(np.int32), bins - 1)
        dq = np.floor((dv + 1) / 2 * bins).astype(np.int32)
        for k in range(len(f)):
            want = sorted(map(tuple, q[f[order[k]]]))
            got = sorted(map(tuple, dq[df[k]]))
            assert want == got, (name, k)


def test_encode_long_strip_is_iterative():
    """200k-face strip: the reference recurses once per face; the native traversal must not depend on stack depth."""
    import meshes
    from meto import Engine
    n = 200_000
    i = np.arange(n + 2)
    v = np.stack([np.linspace(-0.95, 0.95, n + 2), (i % 2) * 0.1, np.zeros(n + 2)], 1).astype(np.float32)
    k = np.arange(n)
    f = np.where((k % 2 == 0)[:, None], np.stack([k, k + 1, k + 2], 1), np.stack([k + 1, k, k + 2], 1)).astype(np.int32)
    tok, order, ftype = Engine(2048).encode(v, f)
    assert len(order) == n and sorted(order.tolist()) == list(range(n))
    assert len(tok) == 4 * n + 6 * (tok == 2).sum()


def test_encode_rejects_bad_indices():
    from meto import Engine
    v = np.zeros((3, 3), np.float32)
    with pytest.raises(ValueError):
        Engine(512).encode(v, np.array([[0, 1, 3]]))
    tok, order, ftype = Engine(512).encode(v, np.zeros((0, 3), np.int32))
    assert len(tok) == 0 and len(order) == 0 and len(ftype) == 0


def test_simple_mesh_clean_up():
    """edgerunner_b200.mesh.SimpleMesh (used by save_mesh when trimesh is absent): merge, de-duplicate, consistent outward winding."""
    import meshes
    from edgerunner_b200.mesh import SimpleMesh
    v, f = meshes.cube()
    soup_v = v[f].reshape(-1, 3)                                   # un-indexed triangle soup, like the detokenizer's output
    soup_f = np.arange(len(soup_v)).reshape(-1, 3)
    soup_f[[1, 4, 7]] = soup_f[[1, 4, 7]][:, ::-1]                 # three faces with the wrong winding
    soup_f = np.concatenate([soup_f, soup_f[:2][:, [1, 2, 0]]])    # two duplicated faces (rotated index order)
    m = SimpleMesh(vertices=soup_v, faces=soup_f)
    m.merge_vertices()
    assert m.vertices.shape == (8, 3)
    m.update_faces(m.unique_faces())
    assert m.faces.shape == (12, 3)
    m.fix_normals()
    assert m.volume == pytest.approx(1.9 ** 3, rel=1e-6)           # closed, consistently wound, outward: +volume of the 1.9 cube
    two = SimpleMesh(vertices=np.concatenate([v, v + 3.0]), faces=np.concatenate([f[:, ::-1], f + len(v)]))
    two.fix_normals()                                              # first component inverted as a whole, second one fine
    assert two.volume == pytest.approx(2 * 1.9 ** 3, rel=1e-6)


# ------------------------------------------------------------------ LR backend (Options.meto_backend = 'LR') ------------------------------------------------------------------

def test_lr_backend_matches_reference_goldens(golden_dir):
    """Engine(backend='LR'): encode + decode against the compiled reference's Engine_LR (residual coordinates, repeated faces, -1 markers)."""
    import meshes
    from meto import Engine
    g = np.load(os.path.join(golden_dir, 'meto.npz'))
    fixtures = dict(meshes.all_meshes())
    fixtures.update(meshes.stress_meshes())
    n = repeated = 0
    for key in list(g['lr_names']) + list(g['lr_enc_names']):
        key = str(key)
        name, bins = key[3:].rsplit('_', 1)
        v, f = fixtures[name]
        eng = Engine(int(bins), backend='LR')
        assert eng.num_tokens == 2 * int(bins) + 3
        tok, order, ftype = eng.encode(v, f)
        np.testing.assert_array_equal(tok, g[key + '_tokens'], err_msg=key)
        np.testing.assert_array_equal(order, g[key + '_order'], err_msg=key)
        np.testing.assert_array_equal(ftype, g[key + '_ftype'], err_msg=key)
        repeated += len(order) != len(f)
        if key + '_dv' in g:
            dv, df, dt = eng.decode(tok)
            np.testing.assert_array_equal(dv, g[key + '_dv'].reshape(-1, 3), err_msg=key)
            np.testing.assert_array_equal(df, g[key + '_df'].reshape(-1, 3), err_msg=key)
            np.testing.assert_array_equal(dt, g[key + '_dt'], err_msg=key)
        n += 1
    assert n >= 60 and repeated > 0          # the capacity-retry path of er_meto_encode is exercised
    for i in range(int(g['n_lr_streams'])):
        dv, df, dt = Engine(512, backend='LR').decode(g[f'lr_stream{i}_tokens'])
        np.testing.assert_array_equal(dv, g[f'lr_stream{i}_dv'].reshape(-1, 3), err_msg=f'stream {i}')
        np.testing.assert_array_equal(df, g[f'lr_stream{i}_df'].reshape(-1, 3), err_msg=f'stream {i}')
        np.testing.assert_array_equal(dt, g[f'lr_stream{i}_dt'], err_msg=f'stream {i}')


def test_clers_backend_matches_reference_goldens(golden_dir):
    """Engine(backend='CLERS'): encode + decode against the compiled reference's Engine_CLERS (EdgeBreaker C/L/E/R/S ops, S-stack, offset
    residuals), every truncation of a two-component stream, and coordinates where an operator is expected."""
    import meshes
    from meto import Engine
    g = np.load(os.path.join(golden_dir, 'meto_clers.npz'))
    fixtures = dict(meshes.all_meshes())
    fixtures.update(meshes.stress_meshes())
    ops = set()
    for key in g['names']:
        key = str(key)
        name, bins = key[len('clers_'):].rsplit('_', 1)
        v, f = fixtures[name]
        eng = Engine(int(bins), backend='CLERS')
        assert eng.num_tokens == 2 * int(bins) + 7
        tok, order, ftype = eng.encode(v, f)
        np.testing.assert_array_equal(tok, g[key + '_tokens'], err_msg=key)
        np.testing.assert_array_equal(order, g[key + '_order'], err_msg=key)
        np.testing.assert_array_equal(ftype, g[key + '_ftype'], err_msg=key)
        dv, df, dt = eng.decode(tok)
        np.testing.assert_array_equal(dv.astype(np.float32), g[key + '_dv'].reshape(-1, 3), err_msg=key)
        np.testing.assert_array_equal(df, g[key + '_df'].reshape(-1, 3), err_msg=key)
        np.testing.assert_array_equal(dt, g[key + '_dt'], err_msg=key)
        ops |= set(np.asarray(ftype).tolist())
    assert len(g['names']) >= 40 and ops == {0, 1, 2, 3, 4}     # every EdgeBreaker op occurs
    eng = Engine(64, backend='CLERS')
    for i in range(int(g['n_streams'])):
        dv, df, dt = eng.decode(g[f'clers_stream{i}_tokens'].astype(np.int64))
        np.testing.assert_array_equal(dv.astype(np.float32), g[f'clers_stream{i}_dv'].reshape(-1, 3), err_msg=f'stream {i}')
        np.testing.assert_array_equal(df, g[f'clers_stream{i}_df'].reshape(-1, 3), err_msg=f'stream {i}')
        np.testing.assert_array_equal(dt, g[f'clers_stream{i}_dt'], err_msg=f'stream {i}')
    # where the reference reads out of bounds this implementation stops: an E as the very last token, an E with nothing to pop
    tok = g['clers_two_components_512_tokens'].astype(np.int64)
    first_e = int(np.flatnonzero(tok == 2)[0])
    dv, df, dt = Engine(512, backend='CLERS').decode(tok[:first_e + 1])
    assert len(df) >= 1 and dt[-1] == 2
    dv, df, dt = Engine(512, backend='CLERS').decode(np.array([5] + [1100] * 9 + [2, 1100, 1100, 1100, 0]))
    assert len(df) == 1


def test_unknown_backend_is_refused():
    from meto import Engine
    with pytest.raises(NotImplementedError):
        Engine(512, backend='EDGEBREAKER')


def test_native_mesh_clean_matches_python_steps():
    """er_mesh_clean (one native call) == SimpleMesh.merge_vertices + update_faces(unique_faces()) + fix_normals, on triangle soups with
    duplicated vertices / faces and random flips; outward orientation gives the positive volume of the closed fixtures."""
    import meshes
    from edgerunner_b200.mesh import SimpleMesh
    rng = np.random.RandomState(4)
    for name in ('cube', 'tetrahedron', 'torus', 'icosphere', 'icosphere2', 'two_components', 'grid', 'annulus'):
        v, f = meshes.all_meshes()[name]
        soup_v = v[f].reshape(-1, 3).astype(np.float64)          # like the detokenizer's output: three fresh vertices per face
        soup_f = np.arange(len(soup_v)).reshape(-1, 3)
        flip = rng.rand(len(soup_f)) < 0.4
        soup_f[flip] = soup_f[flip][:, ::-1]
        soup_f = np.concatenate([soup_f, soup_f[:3][:, [2, 0, 1]]])
        a = SimpleMesh(vertices=soup_v, faces=soup_f)
        a.merge_vertices(); a.update_faces(a.unique_faces()); a.fix_normals()
        b = SimpleMesh(vertices=soup_v, faces=soup_f)
        b.clean_up()
        np.testing.assert_array_equal(a.vertices, b.vertices, err_msg=name)
        assert len(b.faces) == len(f), name
        if name in ('cube', 'tetrahedron', 'torus', 'icosphere', 'icosphere2', 'two_components'):   # closed: orientation is unique
            np.testing.assert_array_equal(a.faces, b.faces, err_msg=name)
            assert b.volume > 0
        else:                                                                       # open patch: consistent up to a global flip
            same = (a.faces == b.faces).all(axis=1)
            assert same.all() or (a.faces[:, ::-1] == b.faces).all(), name
    e = SimpleMesh(vertices=np.zeros((0, 3)), faces=np.zeros((0, 3), dtype=np.int64))
    e.clean_up()
    assert e.vertices.shape == (0, 3) and e.faces.shape == (0, 3)
