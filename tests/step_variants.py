"""The `k_step` instantiations of the library and the parity cases that launch each of them (test infrastructure).

`kStepVariants` in csrc/as_api.cu lists every instantiation `select_step` can choose.  `parse_step_variants` reads its
initialiser rows (counted from 1, in table order); `CASES` is the case table of tests/test_gpu_step_variants.py.  The
CPU suite checks that the cases name every row, so a new instantiation without a case fails there.
"""
from __future__ import annotations

import dataclasses
import os
import re
from typing import Dict, List, Tuple

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AS_API = os.path.join(ROOT, "allsteps_isaaclab_b200", "csrc", "as_api.cu")
TILE = 128  # envs per step-kernel CTA (kTile)
SEPARATE_GATHER_MIN_ENVS = 1 << 16  # kSeparateGatherMinEnvs: from here on k_prepare* gathers for the step kernel

MODE_NUMBERS = {"kModeFused": 0, "kModePass1": 2, "kModePass2": 3}  # StepMode
MODE_NAMES = {"kModeFused": "fused", "kModePass1": "pass1", "kModePass2": "pass2"}
KIND_NAMES = {"kRagged": "ragged", "kRuntimeDiv": "runtime-div", "kTwoFma": "two-fma", "kPrepared": "prepared"}
TEMPLATE_DEFAULTS = (None, None, None, "false", "false", "false")  # k_step<MODE, EXACT, FULL, FAST, PACKED, PRE>

_ROW = re.compile(r"\{\s*(kMode\w+)\s*,\s*(k\w+)\s*,\s*(true|false)\s*,\s*(true|false)\s*,\s*k_step<([^>]*)>\s*\}")
# the demangled name of an instantiation, as the CUDA profiler reports it
KERNEL_NAME = re.compile(r"k_step<(\d+), (\d+), (true|false), (true|false), (true|false), (true|false)>")


@dataclasses.dataclass(frozen=True)
class StepVariant:
    row: int  # 1-based position in kStepVariants
    mode: str  # fused / pass1 / pass2
    kind: str  # ragged / runtime-div / two-fma / prepared
    fast: bool
    packed: bool
    template: Tuple[int, int, bool, bool, bool, bool]  # (MODE, EXACT, FULL, FAST, PACKED, PRE)


def _template(args: str) -> Tuple[int, int, bool, bool, bool, bool]:
    parts = [p.strip() for p in args.split(",")]
    full = parts + list(TEMPLATE_DEFAULTS[len(parts):])
    mode = MODE_NUMBERS[full[0]]
    return (mode, int(full[1]), *(v == "true" for v in full[2:]))


def parse_step_variants(path: str = AS_API) -> List[StepVariant]:
    src = open(path).read()
    body = re.search(r"const StepVariant kStepVariants\[\] = \{(.*?)\n\};", src, re.S)
    assert body, "kStepVariants not found in as_api.cu"
    rows = []
    for i, m in enumerate(_ROW.finditer(body.group(1)), start=1):
        mode, kind, fast, packed, args = m.groups()
        rows.append(StepVariant(i, MODE_NAMES[mode], KIND_NAMES[kind], fast == "true", packed == "true",
                                _template(args)))
    return rows


def parse_kernel_name(name: str):
    m = KERNEL_NAME.search(name)
    if m is None:
        return None
    g = m.groups()
    return (int(g[0]), int(g[1]), *(v == "true" for v in g[2:]))


@dataclasses.dataclass(frozen=True)
class Case:
    """One replay of tests/test_gpu_step_variants.py and the kStepVariants rows it must launch (full-tile row first,
    then the ragged row when N % 128 != 0).

    mode      fused: `mdp.step`; pass1: `pass1` -> `reset` -> `pass2` / `no_reset`; pass2: `reset` + `pass2` with no
              pass 1 open (the order of DirectRLEnv.reset())
    layout    contiguous / isaac (slices of one 16-byte aligned (N,13) root tensor: PACKED) / pinned_contact (contact
              matrices in pinned host memory: a fused step at N >= 65 536 gathers them itself, two-FMA)
    outputs   the generic-instantiation triggers: reward_terms, obs_clip, final_obs, quat_xyzw (none: FAST)
    exact_div one joint range with an all-ones significand: the instantiations that read the division flavour at run time
    """
    name: str
    mode: str
    num_envs: int
    rows: Tuple[int, ...]
    layout: str = "contiguous"
    outputs: Tuple[str, ...] = ()
    exact_div: bool = False

    @property
    def fast(self) -> bool:
        return not self.outputs

    @property
    def packed(self) -> bool:
        return self.layout == "isaac"

    @property
    def prepared(self) -> bool:
        return self.num_envs >= SEPARATE_GATHER_MIN_ENVS and self.layout != "pinned_contact"


CASES = (
    Case("fused-two-fma", "fused", 1001, (3, 1), outputs=("reward_terms",)),
    Case("fused-two-fma-packed", "fused", 1024, (4,), layout="isaac", outputs=("obs_clip",)),
    Case("fused-two-fma-fast", "fused", 1000, (5, 1)),
    Case("fused-two-fma-fast-packed", "fused", 2048, (6,), layout="isaac"),
    Case("fused-two-fma-pinned-contacts", "fused", 65536, (3,), layout="pinned_contact", outputs=("reward_terms",)),
    Case("fused-runtime-div", "fused", 1001, (2, 1), outputs=("reward_terms",), exact_div=True),
    Case("fused-prepared", "fused", 65536 + 44, (7, 1), outputs=("final_obs",)),
    Case("fused-prepared-packed", "fused", 65536, (8,), layout="isaac", outputs=("quat_xyzw", "reward_terms")),
    Case("fused-prepared-fast", "fused", 65536, (9,)),
    Case("fused-prepared-fast-packed", "fused", 65536 + 44, (10, 1), layout="isaac"),
    Case("pass1-runtime-div", "pass1", 1001, (12, 11), outputs=("reward_terms",)),
    Case("pass1-prepared", "pass1", 65536 + 44, (13, 11), outputs=("reward_terms", "final_obs")),
    Case("pass1-prepared-packed", "pass1", 65536, (14,), layout="isaac", outputs=("obs_clip",)),
    Case("pass1-prepared-fast", "pass1", 65536, (15,)),
    Case("pass1-prepared-fast-packed", "pass1", 65536 + 44, (16, 11), layout="isaac"),
    Case("pass2-outside-a-step", "pass2", 1001, (18, 17), outputs=("reward_terms",)),
)


def rows_by_number(variants: List[StepVariant]) -> Dict[int, StepVariant]:
    return {v.row: v for v in variants}
