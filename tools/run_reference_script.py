#!/usr/bin/env python
"""Run an UNMODIFIED script of the reference (train_wgan.py, train_gan.py, train_autoencoder.py, ...) against the drop-in `model`
package of this repository: sys.path = [this repo, the reference], a scratch working directory with a small synthetic `data/` tree,
and `itertools.count` capped so that the script's endless epoch loop ends after --epochs epochs.

    python tools/run_reference_script.py /path/to/reference/train_wgan.py --epochs 1 --samples 96 -- nogui

On a CUDA machine the script trains on libsg_b200; on a CPU-only host it runs up to its first forward pass, where the package
raises its "no CPU fallback" error."""
import argparse
import itertools
import os
import runpy
import sys
import tempfile

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _StopTraining(Exception):
    pass


def make_data(root, samples, seed=0):
    rng = np.random.default_rng(seed)
    for res in (8, 16, 32, 64):
        d = os.path.join(root, 'data', 'chairs', 'voxels_%d' % res)
        os.makedirs(d, exist_ok=True)
        n = samples if res == 32 else min(samples, 8)
        for i in range(n):
            np.save(os.path.join(d, '%04d.npy' % i), (rng.standard_normal((res, res, res)) * 0.05).astype(np.float32))
    with open(os.path.join(root, 'data', 'chairs', 'train.txt'), 'w') as f:
        f.write('\n'.join('%04d' % i for i in range(min(samples, 8))) + '\n')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('script')
    ap.add_argument('--epochs', type=int, default=1)
    ap.add_argument('--samples', type=int, default=96)
    ap.add_argument('--workdir', default=None)
    argv = sys.argv[1:]
    script_args = []
    if '--' in argv:
        cut = argv.index('--')
        argv, script_args = argv[:cut], argv[cut + 1:]
    args = ap.parse_args(argv)
    args.script_args = script_args
    ref = os.path.dirname(os.path.abspath(args.script))
    work = args.workdir or tempfile.mkdtemp(prefix='sg_refscript_')
    make_data(work, args.samples)
    os.chdir(work)
    sys.path[:0] = [REPO, ref]
    real_count = itertools.count

    script_file = os.path.abspath(args.script)

    def capped(start=0, step=1):
        # only the script's own `for epoch in count():` is capped; libraries that use itertools.count keep the real one
        if os.path.abspath(sys._getframe(1).f_code.co_filename) != script_file:
            return real_count(start, step)

        def gen():
            for v in real_count(start, step):
                if v - start >= args.epochs * step:
                    raise _StopTraining()
                yield v
        return gen()
    itertools.count = capped
    sys.argv = [args.script] + list(args.script_args)
    try:
        runpy.run_path(args.script, run_name='__main__')
    except _StopTraining:
        print('[run_reference_script] stopped after %d epoch(s); cwd %s' % (args.epochs, work))
    finally:
        itertools.count = real_count


if __name__ == '__main__':
    main()
