"""CPU (-m "not gpu"): the drop-in contract that needs no GPU — the C-ABI library loads and exports every symbol
include/sg_b200.h declares, module surfaces (names, attributes, state_dict keys/shapes/dtypes, checkpoint paths) match
the reference (SURVEY.md Appendix B/C), and the product path refuses CPU tensors instead of falling back."""
import os
import re

import pytest
import torch

import test_oracle_golden as T      # shape tables pinned against the reference's goldens

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_library_exports_every_declared_symbol():
    from shapegan_b200 import _lib as L
    h = L.lib()
    header = open(os.path.join(REPO, 'include', 'sg_b200.h')).read()
    declared = set(re.findall(r'\b(sg_[a-z0-9_]+)\s*\(', header))
    assert declared, 'no declarations parsed'
    for name in declared:
        assert hasattr(h, name), 'libsg_b200.so does not export %s' % name
    missing = declared - set(L.SYMBOLS)
    assert not missing, 'ctypes table lacks %s' % sorted(missing)
    assert h.sg_abi_version() == 1


def _keys(m):
    return {k: tuple(v.shape) for k, v in m.state_dict().items()}


def test_state_dict_contracts():
    from model.autoencoder import Autoencoder
    from model.gan import Discriminator, Generator
    from model.progressive_gan import Discriminator as ProgD
    from model.sdf_net import SDFNet
    assert _keys(Generator()) == {k: tuple(v) for k, v in T.gen_shapes().items()}
    assert list(_keys(Generator())) == list(T.gen_shapes())
    assert _keys(Discriminator()) == {k: tuple(v) for k, v in T.disc_shapes().items()}
    assert _keys(ProgD()) == {k: tuple(v) for k, v in T.prog_shapes().items()}
    assert list(_keys(ProgD())) == list(T.prog_shapes())
    for variational in (True, False):
        assert _keys(Autoencoder(is_variational=variational)) == {k: tuple(v) for k, v in T.ae_shapes(variational).items()}
        assert list(_keys(Autoencoder(is_variational=variational))) == list(T.ae_shapes(variational))
    assert _keys(SDFNet(device='cpu')) == {k: tuple(v) for k, v in T.sdf_shapes().items()}
    assert _keys(SDFNet(latent_code_size=0, device='cpu')) == {k: tuple(v) for k, v in T.sdf_shapes(0).items()}
    sd = Generator().state_dict()
    assert sd['layers.1.num_batches_tracked'].dtype == torch.int64 and sd['layers.0.weight'].dtype == torch.float32
    assert sum(p.numel() for p in ProgD().parameters()) == 4852449          # parameters() de-duplicates the alias


def test_surface_attributes_and_paths():
    from model import CHECKPOINT_PATH, LATENT_CODE_SIZE, LATENT_CODES_FILENAME, MODEL_PATH
    from model.autoencoder import Autoencoder
    from model.gan import Discriminator, Generator
    from model.progressive_gan import RESOLUTIONS, Discriminator as ProgD
    from model.sdf_net import SDFNet
    assert (MODEL_PATH, LATENT_CODE_SIZE) == ('models', 128)
    assert LATENT_CODES_FILENAME == os.path.join('models', 'sdf_net_latent_codes.to')
    g, d, p = Generator(), Discriminator(), ProgD()
    assert g.filename == 'generator.to' and d.filename == 'discriminator.to' and d.use_sigmoid is True
    assert g.get_filename() == os.path.join('models', 'generator.to')
    assert g.get_filename(epoch=7) == os.path.join(CHECKPOINT_PATH, 'generator-epoch-00007.to')
    assert SDFNet(device='cpu').get_filename(epoch=3, filename='sdf_net_latent_codes.to') == \
        os.path.join(CHECKPOINT_PATH, 'sdf_net_latent_codes-epoch-00003.to')
    assert RESOLUTIONS == [8, 16, 32, 64] and p.iteration == 0 and p.fade_in_progress == 1
    p.set_iteration(2)
    assert p.filename == 'hybrid_progressive_gan_discriminator_2.to'
    assert Autoencoder().filename == 'variational-autoencoder-128.to'
    assert Autoencoder(is_variational=False).filename == 'autoencoder-128.to'
    g.filename = 'wgan-generator.to'                     # scripts overwrite it (train_wgan.py:27)
    assert g.get_filename() == os.path.join('models', 'wgan-generator.to')


def test_save_load_roundtrip(tmp_path, monkeypatch):
    from model.sdf_net import SDFNet
    monkeypatch.chdir(tmp_path)
    os.makedirs('models')
    a, b = SDFNet(device='cpu'), SDFNet(device='cpu')
    a.save()
    a.save(epoch=5)
    assert os.path.exists(os.path.join('models', 'checkpoints', 'sdf_net-epoch-00005.to'))
    b.load()
    for (ka, va), (kb, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)
    # the reference's shipped checkpoint format (16 fp32 tensors) loads strictly
    from conftest import load_golden
    g = load_golden('sdfnet_chairs')
    b.load_state_dict({k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith('w.')}, strict=True)


def test_no_cpu_fallback():
    from model.gan import Discriminator, Generator
    from model.sdf_net import SDFNet
    if torch.cuda.is_available():
        pytest.skip('CPU-only check')
    with pytest.raises(RuntimeError, match='CUDA'):
        Discriminator()(torch.zeros(2, 32, 32, 32))
    with pytest.raises(RuntimeError, match='CUDA'):
        Generator()(torch.zeros(2, 128))
    with pytest.raises(RuntimeError, match='CUDA'):
        SDFNet(device='cpu')(torch.zeros(5, 3), torch.zeros(5, 128))


def test_default_init_matches_reference_under_same_seed(tmp_path):
    """Same constructor order => same RNG consumption => identical default-initialised weights.  The reference's digests were
    recorded from its checkout by oracle/init_hashes.py."""
    import json
    import subprocess
    import sys
    with open(os.path.join(REPO, 'tests', 'golden', 'default_init_sha256.json')) as f:
        ref = json.load(f)['sha256']
    r = subprocess.run([sys.executable, os.path.join(REPO, 'oracle', 'init_hashes.py'), REPO], capture_output=True, text=True,
                       cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    ours = json.loads(r.stdout.strip().splitlines()[-1])
    assert ours == ref


def test_sum_arena_slices_are_zeroed_disjoint_and_refreshed():
    """raw.dsums(): reductions take their double workspaces from one memset'ed arena; every slice is handed out once."""
    from shapegan_b200 import raw
    dev = torch.device('cpu')
    arena = raw._SumArena()
    a = arena.take(300, dev)
    b = arena.take(5, dev)
    assert a.dtype == torch.float64 and a.numel() == 300 and b.numel() == 5
    assert a.abs().sum().item() == 0 and b.abs().sum().item() == 0
    a += 1.0
    assert b.abs().sum().item() == 0                                # disjoint
    assert b.data_ptr() - a.data_ptr() == 304 * 8                   # 8-element granularity inside one buffer
    first = arena.buf
    for _ in range(arena.SIZE // 304 + 2):
        c = arena.take(300, dev)
        assert c.abs().sum().item() == 0
    assert arena.buf is not first                                   # exhausted arena replaced by a fresh zeroed one
    big = arena.take(arena.SIZE + 1, dev)
    assert big.numel() == arena.SIZE + 1 and big.abs().sum().item() == 0


def test_splitk_plan_fills_the_machine():
    """sg_igemm_plan (host logic only, no GPU): Conv3d(128->256) on 8^3 -> 4^3 has K = 8192 and few output tiles.  The library picks the
    number of M sub-tiles per CTA together with the K split so that 148 SMs are as full as possible; the workspace it asks for says
    which split it chose: B = 64 -> 32 tiles x 4 splits, B = 128 -> 64 x 2, B = 192 (the batched critic) -> 48 double tiles x 3 splits.
    Layers with at least one wave of tiles are not split."""
    import ctypes
    from shapegan_b200 import _lib as L
    lib = L.lib()

    def plan(mode, b, r, cin, cout, k, out_dims=(0, 0, 0), classes=1):
        a = L.SgIgemmArgs()
        a.mode, a.planes = mode, 1
        a.a = L.SgTensor(ctypes.c_void_p(256), 0, b, r, r, r, cin)
        a.a2 = L.SgTensor(None, 0, 1, 1, 1, 1, 0)
        a.rows = b * (r // 2) ** 3 if mode == L.MODE_CONV else b * r ** 3
        a.k, a.n_pad, a.n_valid = k, cout, cout
        a.b_packed, a.out = ctypes.c_void_p(256), ctypes.c_void_p(256)
        a.out_kind, a.out_ld = L.OUT_BF16, cout
        a.out_d, a.out_h, a.out_w = out_dims
        n = ctypes.c_size_t(0)
        L.check(lib.sg_igemm_plan(ctypes.byref(a), ctypes.byref(n)), 'sg_igemm_plan')
        return n.value, a.rows * classes * cout * 4

    for b, ks in ((64, 4), (128, 2), (192, 3)):
        ws, slab = plan(L.MODE_CONV, b, 8, 128, 256, 64 * 128)
        assert ws == ks * slab, (b, ws / slab)
    ws, _ = plan(L.MODE_CONV, 64, 16, 64, 128, 64 * 64)                      # 256 tiles: more than one wave, no split
    assert ws == 0
    ws, slab = plan(L.MODE_CONVT, 64, 4, 256, 128, 8 * 256, out_dims=(8, 8, 8), classes=8)     # 8 classes x 32 tiles = 256 items: no split
    assert ws == 0
