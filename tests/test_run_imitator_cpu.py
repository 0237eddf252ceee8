"""tests/run_imitator_body.py must be the reference's run_imitator.py main block, character for character, and the lookup
tables of impersonator_b200.mesh must equal the reference's utils/mesh.py ones: both checked against digests of the
reference's own text / outputs, stored by tests/golden/make_run_imitator_golden.py."""
import hashlib
import json
import os

import numpy as np
import pytest

from run_imitator_body import BODY

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "run_imitator.json")
MAPPER = "assets/pretrains/mapper.txt"


def sha256(data):
    return hashlib.sha256(data).hexdigest()


def table_digests(M):
    """Digests of the tables a utils/mesh.py-style module ``M`` builds from the asset files under the cwd (the ones
    models/imitator.py:39-41 and models/swapper.py:34-37 use); 'raises AssertionError' where it refuses."""
    def arr(a):
        return "%s%s:%s" % (a.dtype, a.shape, sha256(np.ascontiguousarray(a).tobytes()))

    def ids(x):
        return sha256(json.dumps(x).encode())
    out = {"mapper.txt": sha256(open(MAPPER, "rb").read())}
    for name in ("uv_seg", "front", "back", "head", "uv", "seg", "par"):
        for fb in (False, True):
            try:
                out["%s fill_back=%d" % (name, fb)] = arr(M.create_mapping(name, MAPPER, contain_bg=True, fill_back=fb))
            except AssertionError:
                out["%s fill_back=%d" % (name, fb)] = "raises AssertionError"
    for fb in (False, True):
        parts = M.get_part_face_ids('par', MAPPER, fill_back=fb)
        out["par ids fill_back=%d" % fb] = ids([[k, [int(i) for i in parts[k]]] for k in parts])
        for kind in ('head_front', 'head_back'):
            out["%s ids fill_back=%d" % (kind, fb)] = ids(sorted(int(i) for i in M.get_part_face_ids(kind, MAPPER, fill_back=fb)))
    return out


def test_body_is_the_reference_main_block():
    assert sha256(BODY.rstrip("\n").encode()) == json.load(open(GOLD))["main_block"]


def test_renderer_tables_from_asset_files(tmp_path, monkeypatch):
    """SMPLRenderer(image_size, tex_size, has_front, fill_back=False) as models/imitator.py:39-41 calls it: faces + lookup
    tables come from the files under assets/pretrains (synthetic files in the real formats here)."""
    from impersonator_b200 import mesh, synthetic as S
    from impersonator_b200.nmr import SMPLRenderer
    S.write_synthetic_assets(str(tmp_path), n_targets=1)
    monkeypatch.chdir(tmp_path)
    r = SMPLRenderer(image_size=256, tex_size=3, has_front=True, fill_back=False)
    assert tuple(r.faces.shape) == (13776, 3) and tuple(r.map_fn.shape) == (13777, 3)
    assert r.map_fn[-1].tolist() == [0.0, 0.0, 1.0] and float(r.map_fn[:-1, 2].abs().max()) == 0.0
    assert float(r.front_map_fn.sum()) == 500.0 and float(r.back_map_fn.sum()) == 700.0      # head minus front
    assert mesh.get_map_fn_dim('uv_seg') == 3
    assert mesh.create_mapping('par', MAPPER, contain_bg=True, fill_back=False).shape == (13776 + 1, 11)
    with pytest.raises(AssertionError):                           # upstream's 'par' table does not support fill_back either
        mesh.create_mapping('par', MAPPER, contain_bg=True, fill_back=True)
    want = json.load(open(GOLD))["tables"]
    got = table_digests(mesh)
    assert got["mapper.txt"] == want["mapper.txt"], "the synthetic mapper.txt differs from the one the reference read"
    assert got == want, sorted(k for k in want if got.get(k) != want[k])


def test_networks_factory_names():
    from impersonator_b200.networks import NetworksFactory, HumanModelRecovery       # noqa: F401
    import pytest as _pt
    with _pt.raises(ValueError):
        NetworksFactory.get_by_name('nope')
    g = NetworksFactory.get_by_name('impersonator', bg_dim=4, src_dim=6, tsf_dim=6, repeat_num=6)
    assert g.n_down == 3 and g.repeat_num == 6
