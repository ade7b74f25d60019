"""B200-native PINN residual-and-gradient hot path for the parametric H2+ model
(arXiv:2211.04607) as implemented by slitvinov/PINN_for_quantum_wavefunction_surfaces.

Only the hot path lives here: the fused loss + parameter-gradient kernels behind a C ABI
(``libpinn_b200.so``, ``include/pinn_b200.h``) and the Python mirror of the reference's
call sites:

* ``PinnLossPoc`` / ``PinnLossTrainPy`` - ``torch.autograd.Function`` replacements of
  ``NN_ion.LossFunctions`` (poc/main.py:341-355) and of the inline block train.py:41-57
* ``HostStep``        - the training evaluation on fixed host buffers, arguments bound once (``pinn_loss_fwd_bwd_host``)
* ``fields``          - fused ``parametricPsi`` + ``hamiltonian`` (poc/main.py:321, 118)
* ``loss_eval``       - the loss without its gradient: a forward-only reduction in float64 (held-out / validation losses)
* ``patch_nn_ion``    - monkey-patches an ``NN_ion`` class so the reference training loop runs unchanged
* ``run_train_py``    - runs the reference ``train.py`` with lines 41-57 routed through the kernel
* ``trainer``         - device-resident loop: Philox sampler, fused Adam, CUDA-graph replay (train.py:21-72; poc/main.py:359-430),
  and a device-resident torch.optim.LBFGS (``Trainer.run_lbfgs``, ``LBFGSState``)
* ``analysis``        - dense-grid energies / Hellmann-Feynman force / E(R) curve (poc/main.py:438-517, 639-676; energy.py)
* ``convert``         - ``model.bin`` and ``.pt`` containers <-> packed parameters

There is no CPU fallback: importing works anywhere, but every compute entry raises if the
CUDA library or a B200 is missing.
"""
from .params import (N_THETA, POC_TENSOR_NAMES, TRAINPY_TENSOR_NAMES, pack_poc, unpack_poc, pack_trainpy,
                     unpack_trainpy, FINE_TUNE_GRAD_MASK)
from ._lib import lib, Handle, PinnError, library_path, bind_host_to_device_numa
from .ops import (PinnLossPoc, PinnLossTrainPy, loss_poc, loss_trainpy, fields, loss_and_grad_raw, loss_eval,
                  indices_to_mask, HostStep)
from .patch import patch_nn_ion, run_train_py, trainpy_patched_source
from . import analysis, convert, trainer
from .trainer import Trainer, AdamState, adam_step, LBFGSState, lbfgs_begin, lbfgs_advance, sample, sample_adaptive, train_trainpy, train_poc, init_trainpy, init_poc

__all__ = [
    "N_THETA", "POC_TENSOR_NAMES", "TRAINPY_TENSOR_NAMES", "pack_poc", "unpack_poc", "pack_trainpy",
    "unpack_trainpy", "FINE_TUNE_GRAD_MASK", "lib", "Handle", "PinnError", "library_path", "bind_host_to_device_numa", "PinnLossPoc",
    "PinnLossTrainPy", "loss_poc", "loss_trainpy", "fields", "loss_and_grad_raw", "loss_eval", "indices_to_mask", "HostStep",
    "patch_nn_ion", "run_train_py", "trainpy_patched_source", "analysis", "convert", "trainer", "Trainer", "AdamState",
    "adam_step", "LBFGSState", "lbfgs_begin", "lbfgs_advance", "sample", "sample_adaptive", "train_trainpy", "train_poc", "init_trainpy", "init_poc",
]
