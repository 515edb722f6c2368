"""CPU checks of the drop-in boundary: libpsg_b200.so loads without a GPU and exports every symbol
include/psg_b200.h declares; the ctypes binding covers the same set; the product refuses to run
without CUDA instead of falling back to the oracle or to stock PyTorch."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HEADER = os.path.join(REPO, "include", "psg_b200.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(psg_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_entry_points():
    names = _declared()
    for must in ("psg_fps", "psg_ball_query", "psg_three_nn", "psg_square_distance", "psg_index_points",
                 "psg_net_forward", "psg_net_backward", "psg_nb_attack", "psg_nu_step", "psg_confusion_matrix"):
        assert must in names
    assert len(names) >= 40


def test_library_loads_and_exports_every_declared_symbol():
    from pointsecguard_b200 import _lib as L
    lib = ctypes.CDLL(L.LIB_PATH)
    missing = [n for n in _declared() if not hasattr(lib, n)]
    assert not missing, missing
    assert L.psg_version() >= 100


def test_ctypes_binding_covers_the_header():
    from pointsecguard_b200 import _lib as L
    declared, bound = set(_declared()), set(L.EXPORTS)
    assert declared == bound, (sorted(declared - bound), sorted(bound - declared))


def test_header_is_plain_c():
    """The boundary is a C ABI: the header must compile as C with no CUDA / torch headers."""
    import subprocess
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "t.c")
        open(src, "w").write('#include "psg_b200.h"\nint main(void){ return psg_nu_scratch_floats(1, 1) == 0; }\n')
        subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.dirname(HEADER), src])


def test_argument_errors_are_status_codes_not_crashes():
    from pointsecguard_b200 import _lib as L
    # host-side validation happens before anything touches the device
    assert L._cdll.psg_net_workspace(None, 1, 1, 1) == 0
    with pytest.raises(L.PsgError):
        L.psg_fps(None, 1, 1, 16, 4, None, None, None, None, 0, None)
    with pytest.raises(L.PsgError):
        L.psg_net_forward(None, 0, None, None, None)
    with pytest.raises(L.PsgError):
        L.psg_nu_step(None, None, 0, 0, -1, 10, 0.1, 0.0, 1.0, 0.01, 1.0, 0, 4096.0, 0.07, 0, 0, None, None)
    # names that are not library switches
    for name in (b"no_such_option", b"sm_cap", b"dbg"):
        assert L._cdll.psg_set_option(name, 1) == L.PSG_EINVAL


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    from pointsecguard_b200 import synthetic as syn, torchattacks
    from pointsecguard_b200.models import pointnet_util as PU
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    m = get_model(13)
    m.load_state_dict(syn.make_state_dict("ssg"))
    m.eval()
    x = syn.make_blocks(1, 256, 0)
    with pytest.raises(RuntimeError):
        m(x)
    with pytest.raises(RuntimeError):
        torchattacks.NB_attack(m, iters=1)(x, np.zeros((1, 256)))
    with pytest.raises((NotImplementedError, RuntimeError)):
        PU.farthest_point_sample(x[:, :3].permute(0, 2, 1).contiguous(), 16)
    with pytest.raises(RuntimeError):
        PU.PointNetSetAbstraction(16, 0.2, 32, 12, [16], False).eval()(x[:, :3], x)


def test_state_dict_keys_match_the_reference_checkpoint_contract():
    """SURVEY.md section 5: 156 tensors (SSG) / 240 (MSG) with the reference's names and shapes."""
    from pointsecguard_b200 import synthetic as syn
    from pointsecguard_b200.models import pointnet2_sem_seg as S, pointnet2_sem_seg_msg as M
    for mod, arch, n in ((S, "ssg", 156), (M, "msg", 240)):
        sd = mod.get_model(13).state_dict()
        ref = syn.make_state_dict(arch)
        assert len(sd) == n and set(sd.keys()) == set(ref.keys())
        assert all(tuple(sd[k].shape) == tuple(ref[k].shape) for k in sd)
    assert S.get_model(13).sa1.mlp_convs[0].weight.shape == (32, 12, 1, 1)
    assert M.get_model(13).sa1.conv_blocks[1][2].weight.shape == (64, 32, 1, 1)


def test_bn_folding_matches_conv_bn_eval():
    from pointsecguard_b200.engine import fold_conv_bn
    torch.manual_seed(0)
    conv, bn = torch.nn.Conv1d(7, 5, 1), torch.nn.BatchNorm1d(5)
    bn.running_mean.normal_(); bn.running_var.uniform_(0.5, 2); bn.weight.data.uniform_(0.5, 1.5); bn.bias.data.normal_()
    bn.eval()
    x = torch.randn(3, 7, 11)
    w, b = fold_conv_bn(conv.weight, conv.bias, {"weight": bn.weight, "bias": bn.bias, "running_mean": bn.running_mean,
                                                 "running_var": bn.running_var}, bn.eps)
    y = torch.einsum("oc,bcn->bon", torch.from_numpy(w), x) + torch.from_numpy(b)[None, :, None]
    torch.testing.assert_close(y, bn(conv(x)), rtol=1e-5, atol=1e-5)


def test_bare_name_drop_in_imports():
    """The reference's scripts put models/ and attacks/ on sys.path and import by bare name
    (NB_nontarget_test_semseg.py:18-20, 33, 100-103); the package offers the same names under those directories."""
    import subprocess
    import sys
    pkg = os.path.join(REPO, "pointsecguard_b200")
    code = (
        "import sys, importlib\n"
        f"sys.path.insert(0, {REPO!r}); sys.path.append({os.path.join(pkg, 'models')!r}); sys.path.append({pkg!r})\n"
        "MODEL = importlib.import_module('pointnet2_sem_seg'); MSG = importlib.import_module('pointnet2_sem_seg_msg')\n"
        "import torchattacks\n"
        "assert 'pointsecguard_b200' in MODEL.__file__ and 'pointsecguard_b200' in torchattacks.__file__\n"
        "m = MODEL.get_model(13); MSG.get_model(13); MODEL.get_loss()\n"
        "for n in ('NB_attack', 'NU_attack', 'tar_NB_attack', 'tar_NU_attack'):\n"
        "    getattr(torchattacks, n)(m)\n"
        "import pointnet_util as PU\n"
        "for n in ('square_distance', 'index_points', 'farthest_point_sample', 'query_ball_point', 'sample_and_group',\n"
        "          'sample_and_group_all', 'PointNetSetAbstraction', 'PointNetSetAbstractionMsg', 'PointNetFeaturePropagation'):\n"
        "    assert hasattr(PU, n), n\n"
        "print('ok')\n")
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and p.stdout.strip().endswith("ok"), p.stderr[-2000:]
