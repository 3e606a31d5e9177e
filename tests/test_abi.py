"""The C-ABI library builds, loads, and exports exactly what include/fragnet_b200.h declares (CPU only:
no kernel is launched here)."""
import os
import re

from conftest import ROOT


def _declared():
    text = open(os.path.join(ROOT, "include", "fragnet_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fnb_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    from fragnet_b200 import _abi
    assert _declared() == sorted(_abi.SIGNATURES)


def test_library_exports_every_symbol():
    from fragnet_b200 import _abi
    lib = _abi.load()
    for name in _declared():
        assert hasattr(lib, name), name
    assert lib.fnb_version() == _abi.ABI_VERSION
    assert lib.fnb_scratch_bytes() >= 148 * (128 * 256 + 128) * 4
    assert lib.fnb_csr_workspace_bytes(1000, 5000) > 2 * 1000 * 4 + 2 * 5000 * 4
    assert lib.fnb_error_string(0) == b"ok"
    assert b"NULL" in lib.fnb_error_string(-1)


def test_argument_validation_needs_no_gpu():
    """Negative return codes come from host-side checks before any launch."""
    from fragnet_b200 import _abi
    lib = _abi.load()
    assert lib.fnb_csr_build(None, None, -1, 4, 0, None, None, None, None, None, None, None, None, None, 0, None, None) == -2
    assert lib.fnb_csr_build(None, None, 0, 4, 0, None, None, None, None, None, None, None, None, None, 0, None, None) == -1
    assert lib.fnb_proj_fwd(None, None, None, 8, 128, None, 0, 0, 0, None, None, 0, None) == -1
    assert lib.fnb_dropout_relu_fwd(None, None, 4, 1.5, 1, 1, 0, 0, None) == -2
    assert lib.fnb_gat_fwd_tiled(None, None, None) == -1
    assert lib.fnb_gat_bwd_tiled(None, None, None) == -1
    assert lib.fnb_arena_assemble(None, 4, 10, None, 1, None, 0, None, 0, None, None) == -1
    assert lib.fnb_arena_assemble(None, 4, 10, None, 99, None, 0, None, 0, None, None) == -2
    assert lib.fnb_arena_workspace_bytes(1024, 20) >= 20 * (2 * 1024 + 1) * 8


def test_no_cpu_fallback_in_product_path():
    """The product package never imports the oracle."""
    pkg = os.path.join(ROOT, "fragnet_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in re.sub(r'""".*?"""', "", src, flags=re.S), os.path.join(dirpath, f)


def test_ctypes_structs_match_the_header_layout(tmp_path):
    """sizeof / offsetof of every struct in include/fragnet_b200.h, compiled with gcc, equal the ctypes mirrors."""
    import ctypes as C
    import subprocess

    from fragnet_b200 import _abi as A
    pairs = [("fnb_graph", A.CGraph), ("fnb_post_act", A.CPostAct), ("fnb_gat_fwd_args", A.CGatFwdArgs),
             ("fnb_gat_bwd_args", A.CGatBwdArgs), ("fnb_layer_params", A.CLayerParams),
             ("fnb_layer_grads", A.CLayerGrads), ("fnb_batch_plan", A.CBatchPlan), ("fnb_batch_inputs", A.CBatchInputs),
             ("fnb_encoder_opts", A.CEncoderOpts), ("fnb_encoder_io", A.CEncoderIO), ("fnb_mlp3_params", A.CMlp3),
             ("fnb_mlp3_grads", A.CMlp3), ("fnb_pretrain_head_params", A.CPretrainHeadParams),
             ("fnb_pretrain_head_grads", A.CPretrainHeadParams), ("fnb_pretrain_head_io", A.CPretrainHeadIO),
             ("fnb_mse_term", A.CMseTerm), ("fnb_pretrain_step_args", A.CPretrainStepArgs),
             ("fnb_arena_kind", A.CArenaKind), ("fnb_arena_job", A.CArenaJob), ("fnb_widen_job", A.CWidenJob), ("fnb_peer_set", A.CPeerSet)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "fragnet_b200.h"', 'int main(void){']
    for cname, cls in pairs:
        lines.append(f'printf("{cname} %zu", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'printf(" %zu", offsetof({cname}, {fname}));')
        lines.append('printf("\\n");')
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.strip().splitlines()
    for (cname, cls), line in zip(pairs, out):
        got = [int(x) for x in line.split()[1:]]
        want = [C.sizeof(cls)] + [getattr(cls, f).offset for f, _ in cls._fields_]
        assert got == want, cname


def test_fragnet_shim_falls_through_to_a_reference_checkout(tmp_path):
    """The ``fragnet`` shim serves the hot path; with the reference further down sys.path, modules and names outside
    it are the reference's own (pretrain_gat2.py:4-12 imports ``fragnet.dataset.dataset.load_data_parts`` and
    ``FragNetPreTrainMasked`` next to the classes the shim replaces)."""
    import os
    import subprocess
    import sys
    ref = tmp_path / "ref"
    (ref / "fragnet" / "dataset").mkdir(parents=True)
    (ref / "fragnet" / "model" / "gat").mkdir(parents=True)
    (ref / "fragnet" / "dataset" / "dataset.py").write_text("def load_data_parts():\n    return 'reference'\n")
    (ref / "fragnet" / "model" / "gat" / "pretrain_heads.py").write_text(
        "from fragnet.model.gat.gat2 import FragNet\n\n\nclass FragNetPreTrainMasked:\n    encoder = FragNet\n\n\n"
        "class FragNetPreTrain:\n    shadowed = True\n")
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "from fragnet.dataset.dataset import load_data_parts\n"
        "from fragnet.model.gat.pretrain_heads import FragNetPreTrain, FragNetPreTrainMasked\n"
        "import fragnet_b200.model.gat.pretrain_heads as ours, fragnet_b200.model.gat.gat2 as g\n"
        "assert load_data_parts() == 'reference'\n"
        "assert FragNetPreTrain is ours.FragNetPreTrain and not hasattr(FragNetPreTrain, 'shadowed')\n"
        "assert FragNetPreTrainMasked.encoder is g.FragNet\n"
        "import fragnet.model.gat.pretrain_heads as shim\n"
        "try:\n    shim.Nope\n    raise SystemExit('no AttributeError')\n"
        "except AttributeError as e:\n    assert 'hot path' in str(e)\n"
        "print('ok')\n")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([repo, str(ref)]))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=str(tmp_path))
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]
