"""dftatom_b200 — B200-native radial Kohn-Sham SCF engine (host-side Python mirror of the reference interface).

The product is `libdftatom_b200.so` (CUDA sm_100a kernels behind the C ABI of include/dftatom_b200.h); this
package is a thin ctypes binding over that ABI plus a mirror of the reference's entry points
(`DFT::DFTAtom::CalculateNonUniformLDA/LSDA`, reference DFTAtom/DFTAtom.h:14,17, and `Options`,
Options.h:48-54).  There is no CPU fallback: importing works anywhere, but creating a `Context` without the
built extension or without a CUDA device raises.
"""
from .api import (  # noqa: F401
    Context,
    DFTAtom,
    DFTAtomError,
    KleinmanBylander,
    Level,
    LogDerivatives,
    Options,
    PartialCore,
    Pseudopotential,
    Radial,
    Result,
    Step,
    aufbau,
    config_aufbau,
    estimate_cost,
    format_config,
    lib_path,
    load_library,
    n_nodes,
    orbital_count,
    parse_config,
    partition,
    split_spin,
)
from .report import format_report, parse_report  # noqa: F401

__all__ = [
    "Context", "DFTAtom", "DFTAtomError", "KleinmanBylander", "Level", "LogDerivatives", "Options", "PartialCore", "Pseudopotential", "Radial", "Result", "Step", "aufbau", "split_spin", "n_nodes",
    "lib_path", "load_library", "format_report", "parse_report", "estimate_cost", "partition", "orbital_count",
    "config_aufbau", "parse_config", "format_config",
]
