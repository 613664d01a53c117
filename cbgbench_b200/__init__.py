"""cbgbench_b200 - B200-native implementation of CBGBench's diffusion-sampling hot path.

Only what the path needs (DESIGN.md):
  csrc/         hand-written sm_100a CUDA kernels + the C-ABI (include/cbg_b200.h)
  modules.py    nn.Module mirror of the reference denoiser (same signatures / state-dict keys)
  targetdiff.py TargetDiff.sample drop-in (outer diffusion loop in Python, one C call per step)
  diffsbdd.py   DiffSBDD.sample drop-in (row f2: variational schedule + COM projection on the same denoiser)
  diffbp.py     DiffBP.sample drop-in (row f2: CoM head = 3 more H2X layers, score-form VP step, mask-type step)
  difffg.py     D3FG.sample drop-in (FG context embedder, IPA encoder, position / SO(3) / FG-type reverse step)
  schedulers.py noise-schedule tables (checkpoint-compatible parameter containers)
  sharding.py   pocket sharding over GPUs + the single gather of final coordinates
  batch_builder.py  sampling batches built on the GPU from raw pockets (row f3: size prior, types, positions, collate)
  sample_driver.py  sample.py-style loop (row f1)
  synthetic.py  synthetic pockets / seeded weights for tests and benchmarks

There is no CPU or PyTorch fallback: compute entry points raise if libcbg_b200.so is missing.
"""
from .modules import UniTransformerB200, get_e3_gnn  # noqa: F401
from .targetdiff import TargetDiffB200, get_model, register_model  # noqa: F401
from .diffsbdd import DiffSBDDB200  # noqa: F401
from .diffbp import DiffBPB200  # noqa: F401
from .difffg import D3FGB200  # noqa: F401
from .batch_builder import DeviceBatchBuilder, SizePrior  # noqa: F401

__version__ = '0.1.0'
