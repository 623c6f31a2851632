"""Resolves every python config the reference ships (configs/**/*.py, `_base_` inheritance followed by ssdnerf_b200.Config, the same
semantics as mmcv.Config) and stores the parts the hot paths consume -- `model`, `train_cfg`, `test_cfg`, `data.samples_per_gpu` --
as tests/golden/reference_configs.json.  Run as `REF=<checkout of the reference> python tests/golden/make_config_fixtures.py`;
bench.py and the tests build their models from this fixture: the reference's own settings, not a restatement."""
import glob
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
REF = os.environ.get('REF', '')


def plain(x):
    if isinstance(x, dict):
        return {k: plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [plain(v) for v in x]
    return x


def resolve_all():
    from ssdnerf_b200 import Config
    if not REF or not os.path.isdir(os.path.join(REF, 'configs')):
        raise SystemExit(f'REF={REF!r} is not a checkout of the reference (set REF to one)')
    out = {}
    for path in sorted(glob.glob(os.path.join(REF, 'configs', '**', '*.py'), recursive=True)):
        cfg = Config.fromfile(path)
        if 'model' not in cfg:
            continue
        rel = os.path.relpath(path, REF)
        out[rel] = dict(model=plain(cfg['model']), train_cfg=plain(cfg.get('train_cfg', {})), test_cfg=plain(cfg.get('test_cfg', {})),
                        samples_per_gpu=cfg.get('data', {}).get('samples_per_gpu'))
    return out


if __name__ == '__main__':
    cfgs = resolve_all()
    with open(os.path.join(HERE, 'reference_configs.json'), 'w') as f:
        json.dump(cfgs, f, indent=1, sort_keys=True)
    print(len(cfgs), 'configs')
