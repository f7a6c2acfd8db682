"""TEST INFRASTRUCTURE — never imported by the product package.

Imports the UNMODIFIED reference (OpenDriveLab/ST-P3 @ /root/reference) on CPU by
stubbing the third-party packages that are absent from this image (SURVEY.md §8c).
Only usable where /root/reference exists (the build container); the GPU box does
not have it, so everything produced with this loader is shipped as fixtures under
tests/golden/ (see oracle/make_golden.py).

Nothing from the reference is copied: the modules are imported from where they lie.
"""
import os
import sys
import types
from types import SimpleNamespace

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the reference checkout named by STP3_REFERENCE_ROOT, else its unmodified install under the git-ignored oracle/_ref/
# (oracle/build_ref.py)
_CANDIDATES = [os.environ.get("STP3_REFERENCE_ROOT"), os.path.join(_REPO, "oracle", "_ref")]
REFERENCE_ROOT = next((c for c in _CANDIDATES if c and os.path.isdir(os.path.join(c, "stp3"))), _CANDIDATES[-1])


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "stp3"))


def _stub(name, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []  # behave like a package so that sub-imports resolve
    sys.modules[name] = m
    return m


def install_stubs():
    import torch.nn as nn
    import numpy as np

    class _Dummy:  # placeholder class for names the hot path never touches
        def __init__(self, *a, **k):
            pass

    class _DropPath(nn.Module):  # timm.models.layers.DropPath: identity at p=0 / eval
        def __init__(self, p=0.0):
            super().__init__()

        def forward(self, x):
            return x

    class _EfficientNet:  # efficientnet_pytorch.EfficientNet: trunk is injected in tests
        @staticmethod
        def from_pretrained(name):
            raise RuntimeError("EfficientNet trunk is third-party and absent (SURVEY §8c)")

    _stub("pyquaternion", Quaternion=_Dummy)
    _stub("nuscenes")
    _stub("nuscenes.nuscenes", NuScenes=_Dummy)
    _stub("nuscenes.utils")
    _stub("nuscenes.utils.geometry_utils", transform_matrix=lambda *a, **k: None)
    _stub("nuscenes.utils.data_classes", LidarPointCloud=_Dummy, Box=_Dummy)
    _stub("nuscenes.utils.splits", create_splits_scenes=lambda: {})
    _stub("nuscenes.map_expansion")
    _stub("nuscenes.map_expansion.map_api", NuScenesMap=_Dummy)
    _stub("timm")
    _stub("timm.models")
    _stub("timm.models.layers", DropPath=_DropPath)
    _stub("efficientnet_pytorch", EfficientNet=_EfficientNet)
    _stub("skimage")
    _stub("skimage.draw", polygon=lambda *a, **k: None)
    mpl = _stub("matplotlib", use=lambda *a, **k: None)
    _stub("matplotlib.pyplot")
    _stub("matplotlib.pylab")
    mpl.pyplot = sys.modules["matplotlib.pyplot"]
    _stub("pytorch_lightning", LightningModule=object)
    _stub("fvcore")
    _stub("fvcore.common")
    _stub("fvcore.common.config", CfgNode=dict)
    if not hasattr(np, "int"):  # encoder.py:28 uses np.int (removed in numpy >= 1.24)
        np.int = int


def load_reference():
    """Returns a namespace with the reference's hot-path modules."""
    if not reference_available():
        raise RuntimeError(f"reference not present at {REFERENCE_ROOT}")
    install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import stp3.utils.geometry as geometry
    import stp3.utils.network as network
    import stp3.layers.convolutions as convolutions
    import stp3.layers.temporal as temporal
    import stp3.models.temporal_model as temporal_model
    import stp3.models.decoder as decoder
    import stp3.models.encoder as encoder
    import stp3.models.stp3 as stp3_model

    return SimpleNamespace(geometry=geometry, network=network, convolutions=convolutions,
                           temporal=temporal, temporal_model=temporal_model, decoder=decoder,
                           encoder=encoder, stp3=stp3_model)


def make_fake_stp3(ref, x_bound, y_bound, z_bound, d_bound, final_dim, downsample, discount=0.5):
    """A SimpleNamespace carrying exactly the attributes the reference's lift-splat methods
    read (stp3/models/stp3.py:20-32,111-130), so that STP3.create_frustum / get_geometry /
    projection_to_birds_eye_view can be called UNBOUND without building the whole model
    (STP3.__init__ needs fvcore + the EfficientNet download)."""
    res, start, dim = ref.geometry.calculate_birds_eye_view_parameters(x_bound, y_bound, z_bound)
    cfg = SimpleNamespace(
        IMAGE=SimpleNamespace(FINAL_DIM=tuple(final_dim)),
        LIFT=SimpleNamespace(D_BOUND=list(d_bound)),
    )
    fake = SimpleNamespace(cfg=cfg, bev_resolution=res, bev_start_position=start, bev_dimension=dim,
                           encoder_downsample=downsample, discount=discount)
    fake.frustum = ref.stp3.STP3.create_frustum(fake)
    return fake
