"""ORACLE fixture generator — test infrastructure, NOT product code.

Default-initialised weights under a fixed seed, one SHA-256 digest of the state_dict bytes per module.  The same constructor
order consumes the RNG the same way, so the drop-in `model` package must give the digests of the original project's modules.

    python oracle/init_hashes.py ROOT            print the digests of ROOT/model as JSON
    python oracle/init_hashes.py ROOT --write    store them in tests/golden/default_init_sha256.json

The golden was written from the original project's checkout; tests/test_contract_cpu.py runs this on this repository's root.
Each ROOT needs a fresh process (both trees provide a package named `model`).
"""
import hashlib
import json
import os
import sys
import tempfile
import types

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, 'tests', 'golden', 'default_init_sha256.json')
SEED = 123


def init_hashes(root):
    for n in ('trimesh', 'skimage', 'skimage.measure'):            # imported by model/sdf_net.py, unused by the constructors
        sys.modules.setdefault(n, types.ModuleType(n))
    torch.nn.Module.cuda = lambda self, device=None: self           # the original constructors call self.cuda()
    sys.path.insert(0, root)
    import model.autoencoder as A
    import model.gan as G
    import model.progressive_gan as P
    import model.sdf_net as S
    ctors = {'gan.Generator': G.Generator, 'gan.Discriminator': G.Discriminator, 'progressive_gan.Discriminator': P.Discriminator,
             'autoencoder.Autoencoder': A.Autoencoder,
             'autoencoder.Autoencoder(is_variational=False)': lambda: A.Autoencoder(is_variational=False),
             'sdf_net.SDFNet': lambda: S.SDFNet(device='cpu')}
    out = {}
    for name, ctor in ctors.items():
        torch.manual_seed(SEED)
        sd = ctor().state_dict()
        out[name] = hashlib.sha256(b''.join(v.detach().cpu().numpy().tobytes() for v in sd.values())).hexdigest()
    return out


if __name__ == '__main__':
    root = os.path.abspath(sys.argv[1])
    with tempfile.TemporaryDirectory(prefix='sg_init_') as scratch:
        os.chdir(scratch)                                           # the original util.py creates directories in the cwd on import
        digests = init_hashes(root)
        os.chdir(REPO)
    if '--write' in sys.argv[2:]:
        with open(GOLDEN, 'w') as f:
            json.dump({'_meta': {'seed': SEED, 'torch': torch.__version__,
                                 'what': 'sha256 of the default-initialised state_dict bytes of the original project\'s modules '
                                         '(oracle/init_hashes.py)'},
                       'sha256': digests}, f, indent=1, sort_keys=True)
            f.write('\n')
    print(json.dumps(digests))
