"""cmbpo_b200 -- B200-native model-rollout + GAE path of CMBPO.

Drop-in classes (same constructors / methods as the reference):
    FakeEnv        models/fake_env.py
    ModelSampler   samplers/model_sampler.py
    ModelBuffer    buffers/modelbuffer.py
    CPOBuffer      buffers/cpobuffer.py   (store / finish_path / get)
    B200PE         the model contract of models/base_model.py served by CUDA kernels
    B200Policy     inference side of policies/cpo_policy.py
Everything computes on the GPU through libcmbpo_b200.so (include/cmbpo_b200.h); there is no
CPU fallback.
"""
from . import _lib
from ._lib import CmbpoError, LIB_PATH
from .engine import Engine
from .pe import B200PE
from .policy import B200Policy
from .fake_env import FakeEnv
from .modelbuffer import ModelBuffer
from .cpobuffer import CPOBuffer
from .model_sampler import ModelSampler
from .rollout import RolloutBuffers
from . import statics
from . import dist
from . import checkpoint
from .archive import DeviceArchive
from .checkpoint import load_pe, load_policy, load_state, save_state, write_pe_checkpoint
from . import tf_bundle

__all__ = ["load_pe", "load_policy", "load_state", "save_state", "write_pe_checkpoint", "DeviceArchive", "Engine", "B200PE", "B200Policy", "FakeEnv", "ModelBuffer", "CPOBuffer", "ModelSampler",
           "RolloutBuffers", "CmbpoError", "LIB_PATH", "statics"]
