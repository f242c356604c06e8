"""CPU-only: the oracle/_ref recipe (oracle/make_ref.py).  Where the reference checkout exists (the build container) the vendored
modules must be byte-identical to it; wherever oracle/_ref exists (it travels to the GPU box) the unmodified reference forward must
agree with the oracle port on the same seeded weights — that is what makes `cpu_baseline.kind = "reference"` a statement about the
reference and the oracle a checked restatement of it."""
import hashlib
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"


@pytest.mark.skipif(not os.path.isdir(REF), reason="no reference checkout on this host")
def test_vendored_files_are_the_reference_byte_for_byte(tmp_path):
  sys.path.insert(0, os.path.join(ROOT, "oracle"))
  import make_ref
  assert make_ref.make(REF)
  manifest = json.load(open(os.path.join(make_ref.DST, "MANIFEST.json")))
  assert sorted(manifest) == sorted(make_ref.FILES)
  for rel, digest in manifest.items():
    assert hashlib.sha256(open(os.path.join(REF, rel), "rb").read()).hexdigest() == digest, rel
    assert hashlib.sha256(open(os.path.join(make_ref.DST, rel), "rb").read()).hexdigest() == digest, rel


def test_make_ref_recipe_copies_byte_for_byte_and_records_digests(tmp_path, monkeypatch):
  """The recipe itself, on every host: make() on a stand-in checkout of seeded bytes (CR/LF and non-UTF-8 included) in tmp_path
  copies each module byte for byte and writes both copies' SHA-256 into MANIFEST.json; a missing checkout writes nothing.  It
  says nothing about the reference's contents (the test above does, where a reference checkout exists)."""
  import random
  sys.path.insert(0, os.path.join(ROOT, "oracle"))
  import make_ref
  ref, dst = tmp_path / "reference", tmp_path / "_ref"
  monkeypatch.setattr(make_ref, "DST", str(dst))
  assert not make_ref.make(str(tmp_path / "absent")) and not dst.exists()
  rng = random.Random(0)
  for rel in make_ref.FILES:
    (ref / rel).parent.mkdir(parents=True, exist_ok=True)
    (ref / rel).write_bytes(bytes(rng.randrange(256) for _ in range(rng.randrange(1000, 5000))) + b"\r\n\x00\xff")
  assert make_ref.make(str(ref))
  manifest = json.load(open(dst / "MANIFEST.json"))
  assert sorted(manifest) == sorted(make_ref.FILES)
  for rel, digest in manifest.items():
    assert hashlib.sha256((ref / rel).read_bytes()).hexdigest() == digest, rel
    assert hashlib.sha256((dst / rel).read_bytes()).hexdigest() == digest, rel


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "adaptive_stereo", "models", "stereo_net.py")),
                    reason="oracle/_ref has not been made on this host")
def test_reference_forward_equals_oracle_port():
  code = r'''
import sys
sys.path.insert(0, "%s/oracle")
import torch, stereonet_oracle as O, make_ref
sn = make_ref.load()[0]
fsd, ssd = O.make_feature_state(3, 11), O.make_stereo_state(22, sharpen=40.0)
left, right, _ = O.make_stereo_pair(1, 64, 96, seed=5, max_disp_px=20.0)
f, s = sn.FeatureExtractorNetwork(3), sn.StereoNet(3, 1, 0)
f.load_state_dict(fsd); s.load_state_dict(ssd); f.eval(); s.eval()
with torch.no_grad():
  ref = s(left, f(left), f(right), "l", output_cost_volume=True)
  port = O.predict_disparity_left(fsd, ssd, left, right, 3)
for k, v in port.items():
  err = (ref[k] - v).abs().max().item()
  assert err <= 1e-4, (k, err)
print("OK")
''' % ROOT
  out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
  assert out.returncode == 0 and "OK" in out.stdout, out.stderr[-2000:]
