"""CPU: the drop-in claim of INTEGRATION.md §1 against a record of the UNMODIFIED reference (tests/golden/dropin_imports.json:
what its train.py / eval.py / engine / config import from the packages sigma_b200/dropin replaces, and the config values
train.py builds from).  With `sigma_b200/dropin` FIRST on the path and the dependency stand-ins of `sigma_b200/dropin/shims`
LAST, every recorded import resolves into the drop-in, `models.builder.EncoderDecoder` IS sigma_b200's, and
segmodel(cfg=config, criterion, norm_layer) and AdamW over its parameters construct from the recorded config (train.py:76-93)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r'''
import importlib, json, sys
import torch, torch.nn as nn
rec = json.load(open(sys.argv[2]))
for mod, name, where in rec["imports"]:
    m = importlib.import_module(mod)
    assert m.__file__.startswith(sys.argv[1]), (mod, m.__file__, where)
    assert hasattr(m, name), (mod, name, where)
import sigma_b200.modules as M
from models.builder import EncoderDecoder as segmodel
assert segmodel is M.EncoderDecoder, segmodel
from easydict import EasyDict
config = EasyDict(rec["config"])
criterion = nn.CrossEntropyLoss(reduction="mean", ignore_index=config.background)
import contextlib, io
with contextlib.redirect_stdout(io.StringIO()):
    model = segmodel(cfg=config, criterion=criterion, norm_layer=nn.BatchNorm2d)
opt = torch.optim.AdamW(model.parameters(), lr=config.lr, betas=(0.9, 0.999), weight_decay=config.weight_decay)
n = sum(p.numel() for p in model.parameters())
assert n == rec["n_params"], n
print("DROPIN_OK", type(model).__module__, len(model.state_dict()), n)
'''


def test_recorded_reference_imports_resolve_to_dropin(tmp_path):
    dropin = os.path.join(ROOT, "sigma_b200", "dropin")
    rec = os.path.join(ROOT, "tests", "golden", "dropin_imports.json")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, dropin, os.path.join(dropin, "shims")]))
    r = subprocess.run([sys.executable, "-c", SCRIPT, dropin, rec], capture_output=True, text=True, timeout=600, cwd=str(tmp_path), env=env)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    n_state = json.load(open(rec))["n_state"]
    assert f"DROPIN_OK sigma_b200.modules {n_state}" in r.stdout, r.stdout[-500:]
