"""Drop-in boundary, zero-edit route (SURVEY.md 8b): the UNMODIFIED reference model files import through `compat/mamba_ssm`
(the package INTEGRATION.md 2a tells a maintainer to put on sys.path) and build models whose parameters match the product
mirrors name by name and shape by shape.  CPU only: nothing is launched, the modules are only constructed.
The tests that load the reference model files need the reference tree (REFERENCE_ROOT) and skip without it; the compat package's
own name resolution is checked everywhere."""
import importlib.util
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("REFERENCE_ROOT", "/root/reference")
needs_reference = pytest.mark.skipif(not os.path.isdir(REF), reason="reference tree not present")


@pytest.fixture(scope="module")
def compat_path():
    added = [os.path.join(ROOT, "compat"), ROOT]
    try:
        import timm  # noqa: F401
    except Exception:
        added.append(os.path.join(ROOT, "compat", "_timm_shim"))
    for p in added:
        sys.path.insert(0, p)
    for name in [m for m in sys.modules if m == "mamba_ssm" or m.startswith("mamba_ssm.")]:
        del sys.modules[name]
    yield
    for p in added:
        sys.path.remove(p)
    for name in [m for m in sys.modules if m == "mamba_ssm" or m.startswith("mamba_ssm.") or m.startswith("refcompat_")]:
        del sys.modules[name]
    for name in [m for m in sys.modules if m == "timm" or m.startswith("timm.")]:
        if "_timm_shim" in (getattr(sys.modules[name], "__file__", "") or ""):
            del sys.modules[name]


def _load(rel):
    name = "refcompat_" + rel.replace("/", "_").replace(".py", "")
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def _shapes(m):
    return {k: tuple(v.shape) for k, v in m.state_dict().items()}


def test_compat_names_resolve(compat_path):
    import mamba_ssm.ops.selective_scan_interface as ssi
    import mamba_ssm.ops.triton.ssd_combined as ssd
    from mamba_ssm.distributed.distributed_utils import all_reduce, reduce_scatter
    from mamba_ssm.distributed.tensor_parallel import ColumnParallelLinear, RowParallelLinear
    from mamba_ssm.ops.triton.layernorm_gated import RMSNorm
    from mamba_ssm.ops.triton.selective_state_update import selective_state_update

    from medical_image_classification_b200 import selective_scan_interface as p_ssi
    from medical_image_classification_b200 import ssd_combined as p_ssd
    assert ssi.selective_scan_fn is p_ssi.selective_scan_fn
    assert ssd.mamba_chunk_scan_combined is p_ssd.mamba_chunk_scan_combined
    assert RMSNorm is p_ssd.RMSNormGated
    for dead in (ssd.mamba_split_conv1d_scan_combined, selective_state_update, all_reduce, reduce_scatter,
                 ColumnParallelLinear, RowParallelLinear):
        with pytest.raises(NotImplementedError):
            dead()


@needs_reference
def test_medmamba_imports_and_matches_mirror(compat_path):
    ref = _load("MedMamba.py")
    from medical_image_classification_b200 import selective_scan_interface as p_ssi
    from medical_image_classification_b200.models import medmamba_t
    assert ref.selective_scan_fn is p_ssi.selective_scan_fn        # the call site at MedMamba.py:387,411 now lands in libb200ssm
    torch.manual_seed(0)
    r = ref.VSSM(num_classes=6)                                     # reference defaults = MedMamba-T: depths 2-2-4-2, dims 96-768
    m = medmamba_t(num_classes=6)
    assert _shapes(r) == _shapes(m)
    m.load_state_dict(r.state_dict(), strict=True)


@needs_reference
@pytest.mark.parametrize("rel", ["SSD/MedSSD.py", "CNN_Mamba.py"])
def test_ssd_family_imports_and_matches_mirror(compat_path, rel):
    ref = _load(rel)
    from medical_image_classification_b200 import ssd_combined as p_ssd
    from medical_image_classification_b200.ss2d_ssd import SS2D_with_SSD
    assert ref.mamba_chunk_scan_combined is p_ssd.mamba_chunk_scan_combined
    assert ref.RMSNormGated is p_ssd.RMSNormGated
    torch.manual_seed(0)
    r = ref.SS2D_with_SSD(d_model=32, d_state=16, headdim=16)
    m = SS2D_with_SSD(d_model=32, d_state=16, headdim=16)
    assert _shapes(r) == _shapes(m)
    m.load_state_dict(r.state_dict(), strict=True)
    assert isinstance(r.norm, p_ssd.RMSNormGated)


@needs_reference
def test_medssd_vssm_matches_mirror(compat_path):
    ref = _load("SSD/MedSSD.py")
    from medical_image_classification_b200.models import medssd
    torch.manual_seed(0)
    r = ref.VSSM(num_classes=6, depths=[1, 1, 1, 1], dims=[64, 128, 256, 512], d_state=16)
    m = medssd(num_classes=6, depths=(1, 1, 1, 1), dims=(64, 128, 256, 512), d_state=16)
    assert _shapes(r) == _shapes(m)
    m.load_state_dict(r.state_dict(), strict=True)


@needs_reference
def test_crossmamba_imports_and_matches_mirror(compat_path):
    ref = _load("CrossMamba/CrossMamba_fusion_2b2.py")
    from medical_image_classification_b200.crossmamba import CrossMamba
    torch.manual_seed(0)
    r = ref.CrossMamba(d_model=32, d_state=16, headdim=16)
    m = CrossMamba(d_model=32, d_state=16, headdim=16)
    assert _shapes(r) == _shapes(m)
    m.load_state_dict(r.state_dict(), strict=True)


@needs_reference
def test_medssd_kan_imports_and_matches_mirror(compat_path):
    """BASELINE.json configs[3]: MedSSD_kan (SSD backbone, d_state 16, pykan-style head) through the compat package."""
    ref = _load("MedSSD_kan/MedSSD_kan.py")
    from medical_image_classification_b200.models import medssd_kan
    torch.manual_seed(0)
    r = ref.VSSM(num_classes=6, depths=[1, 1, 1, 1], dims=[64, 128, 256, 512], d_state=16)
    m = medssd_kan(num_classes=6, depths=(1, 1, 1, 1), dims=(64, 128, 256, 512), d_state=16)
    assert _shapes(r) == _shapes(m)
    m.load_state_dict(r.state_dict(), strict=True)
