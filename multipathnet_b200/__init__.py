"""multipathnet_b200 — B200-native (sm_100a) detection forward hot path of
facebookresearch/multipathnet behind the reference's own surface.

Host-side mirror (Python; the reference's host language, Lua/Torch-7, is absent from the
build image — see INTEGRATION.md for the LuaJIT-FFI shim in lua/) of:
  fbcoco.ImageDetect        -> multipathnet_b200.ImageDetect        (ImageDetect.lua)
  nn.Foveal / ContextRegion / BBoxNorm, inn.ROIPooling -> multipathnet_b200.modules
  utils.nms / nms_dense / bbox_vote / convertFrom     -> multipathnet_b200.utils
  fbcoco.Tester_FRCNN:testOne                          -> multipathnet_b200.Tester
  torch.load of .t7 models / proposals (no Torch needed)-> multipathnet_b200.t7
  test_runner.lua's replica threads (K per GPU)        -> multipathnet_b200.ModelReplicas
All compute happens in libmpn_b200.so (hand-written CUDA); nothing here falls back to CPU.
"""
from ._lib import (Context, Model, ModelSpec, MpnError, load_library, LIB_PATH,  # noqa: F401
                   MPN_MAX_DET, MPN_REC_FLOATS, MPN_DIST_ID_BYTES, MPN_MAX_BATCH)
from . import models, modules, t7, utils, workloads  # noqa: F401
from .image_detect import ImageDetect  # noqa: F401
from .tester import Tester  # noqa: F401
from .replicas import ModelReplicas  # noqa: F401
