"""Host-side checks of electron configurations (dftatom_config_aufbau, the string form, the ctypes mirrors, the CLI flags) and of the
oracle's configured SCF (orc_scf_config), including Janak's theorem on the oracle.  No GPU needed."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import pytest

import dftatom_b200 as D
import oracle_config_lib as OC
import oracle_lib as O
from dftatom_b200.api import _CConfig, _COccupation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = dict(levels=10, delta=0.004, max_r=15.0, mixing=0.5)      # the small-atom grid of tests/golden/small.json


def _aufbau4(Z, method):
    """The reference's levels (dftatom_aufbau / dftatom_split_spin) as (n, l, spin, occ): alpha then beta, each in (n, l) order."""
    if method & 1:
        a, b, _, _ = D.split_spin(Z)
        return [(L.n, L.l, 0, float(L.occ)) for L in a] + [(L.n, L.l, 1, float(L.occ)) for L in b]
    return [(L.n, L.l, 0, float(L.occ)) for L in D.aufbau(Z)]


def _as4(cfg):
    return [e if len(e) == 4 else (e[0], e[1], 0, e[2]) for e in cfg]


def test_config_aufbau_without_charge_is_the_reference_aufbau():
    for Z in range(1, 119):
        for m in (0, 1, 2, 3):
            assert _as4(D.config_aufbau(Z, m, 0.0)) == _aufbau4(Z, m), (Z, m)


# (Z, charge) -> LDA configuration without the core, documented in include/dftatom_b200.h
IONS = {
    (26, 2): "[Ar] 3d6",             # Fe2+
    (24, 1): "[Ar] 3d4 4s1",         # Cr+ (the reference's Cr is 3d4 4s2)
    (29, 1): "[Ar] 3d9 4s1",         # Cu+ (the reference's Cu is 3d9 4s2)
    (11, 1): "[Ne]",                 # Na+
    (58, 3): "[Kr] 4d10 4f1 5s2 5p6",  # Ce3+
    (8, -1): "[He] 2s2 2p5",         # O-
    (17, -1): "[Ne] 3s2 3p6",        # Cl-
    (10, -1): "[Ne] 3s1",            # Ne-
    (6, 0.5): "[He] 2s2 2p1.5",      # a fractional cation
    (9, -0.25): "[He] 2s2 2p5.25",   # a fractional anion
}


@pytest.mark.parametrize("Z,charge", sorted(IONS))
def test_charge_rule(Z, charge):
    want = D.parse_config(IONS[(Z, charge)], 0)
    assert D.config_aufbau(Z, 0, charge) == want
    # LSDA: every subshell total split like split_spin - alpha min(occ, 2l + 1), beta the rest, listed when nonzero
    split = []
    for n, l, occ in want:
        split.append((n, l, 0, min(occ, 2 * l + 1.0)))
    for n, l, occ in want:
        if occ - min(occ, 2 * l + 1.0) > 0:
            split.append((n, l, 1, occ - min(occ, 2 * l + 1.0)))
    assert D.config_aufbau(Z, 1, charge) == split
    assert sum(e[-1] for e in want) == pytest.approx(Z - charge, abs=1e-12)


def test_charge_rule_rejects_out_of_range():
    for Z, q in ((11, 11), (11, 12.5), (8, -2.5), (0, 0), (119, 0)):
        with pytest.raises(D.DFTAtomError, match="error -2"):
            D.config_aufbau(Z, 0, q)


def test_parse_config():
    assert D.parse_config("1s2 2s2 2p4.5", 0) == [(1, 0, 2.0), (2, 0, 2.0), (2, 1, 4.5)]
    assert D.parse_config("[Ne] 3s1 3p0", 0) == D.config_aufbau(10, 0) + [(3, 0, 1.0), (3, 1, 0.0)]
    for core, Z in (("He", 2), ("Ne", 10), ("Ar", 18), ("Kr", 36), ("Xe", 54), ("Rn", 86)):
        for m in (0, 1):
            assert D.parse_config(f"[{core}]", m) == D.config_aufbau(Z, m)
    # a subshell given again replaces the core's: the excited neon
    assert D.parse_config("[Ne] 2p5 3s1", 0) == [(1, 0, 2.0), (2, 0, 2.0), (2, 1, 5.0), (3, 0, 1.0)]
    # LSDA: totals split like split_spin, or alpha / beta
    assert D.parse_config("[He] 2s2 2p4", 1) == [(1, 0, 0, 1.0), (2, 0, 0, 1.0), (2, 1, 0, 3.0), (1, 0, 1, 1.0), (2, 0, 1, 1.0), (2, 1, 1, 1.0)]
    assert D.parse_config("1s1/1 2s1/0 2p3/0.5", 1) == [(1, 0, 0, 1.0), (2, 0, 0, 1.0), (2, 1, 0, 3.0), (1, 0, 1, 1.0), (2, 0, 1, 0.0),
                                                        (2, 1, 1, 0.5)]
    for bad, m in (("2x3", 0), ("2p", 0), ("[Q]", 0), ("2p3/1", 0), ("[Zz] 2s1", 1)):
        with pytest.raises(D.DFTAtomError):
            D.parse_config(bad, m)


@pytest.mark.parametrize("method", [0, 1])
def test_parse_config_round_trips(method):
    cases = [D.config_aufbau(Z, method, q) for Z, q in ((26, 2), (29, 1), (8, -1), (6, 0.5), (92, 0), (10, -0.3))]
    cases.append(D.parse_config("1s2 2s2 2p4.5 3d0", method))
    if method:
        cases.append(D.parse_config("[Ne] 3s1/0 3p0.25/0.75", 1))
    for c in cases:
        assert D.parse_config(D.format_config(c, method), method) == c


def test_options_configuration_forms():
    assert D.Options(26, charge=2).entries() == [(n, l, 0, o) for n, l, o in D.config_aufbau(26, 0, 2)]
    assert D.Options(10, config="[He] 2s2 2p5 3s1").entries() == [(1, 0, 0, 2.0), (2, 0, 0, 2.0), (2, 1, 0, 5.0), (3, 0, 0, 1.0)]
    assert D.Options(10, config=[(1, 0, 2), (2, 0, 2), (2, 1, 6)]).entries() == [(1, 0, 0, 2.0), (2, 0, 0, 2.0), (2, 1, 0, 6.0)]
    assert D.Options(10).entries() is None
    # positional construction of the reference's six fields is unchanged
    o = D.Options(18, 14, 25.0, 0.0005, 0.5, 1)
    assert (o.Z, o.method, o.charge, o.config) == (18, 1, 0.0, None)
    with pytest.raises(D.DFTAtomError, match="not both"):
        D.Options(10, charge=1, config="[He] 2s2 2p5").entries()
    with pytest.raises(D.DFTAtomError):
        D.Options(10, method=1, config=[(1, 0, 2)]).entries()          # LSDA entries carry a spin
    assert D.orbital_count(19, 0, config="[Ar] 4s1 3d0 4p0") == 8
    assert D.orbital_count(26, 1, charge=3) == len(D.config_aufbau(26, 1, 3))
    assert D.orbital_count(26, 1) == len(_aufbau4(26, 1))


def _layout(struct_name, ctype, extra_fields=()):
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in ctype._fields_]
    src = "#include <stddef.h>\n#include <stdio.h>\n#include \"dftatom_b200.h\"\nint main(void) {\n"
    src += f'    printf("%zu\\n", sizeof({struct_name}));\n'
    for f in fields:
        src += f'    printf("%zu\\n", offsetof({struct_name}, {f}));\n'
    src += "    return 0;\n}\n"
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "layout.c"), "w") as fh:
            fh.write(src)
        exe = os.path.join(tmp, "layout")
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(tmp, "layout.c")], check=True)
        vals = [int(v) for v in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == C.sizeof(ctype), struct_name
    assert vals[1:] == [getattr(ctype, f).offset for f in fields], struct_name


def test_ctypes_config_matches_the_c_layout():
    _layout("dftatom_occupation", _COccupation)
    _layout("dftatom_config", _CConfig)
    assert C.sizeof(_COccupation) == C.sizeof(OC.OrcOrbital) and C.sizeof(_CConfig) == C.sizeof(OC.OrcConfig)


def test_library_exports_the_configuration_entry_points():
    lib = D.load_library()
    assert hasattr(lib, "dftatom_solve_batch_config") and hasattr(lib, "dftatom_config_aufbau")


def test_cli_help_names_the_configuration_flags():
    exe = os.path.join(ROOT, "bin", "dftatom")
    if not os.path.exists(exe):
        pytest.skip("bin/dftatom not built")
    out = subprocess.run([exe, "--help"], check=True, capture_output=True, text=True).stdout
    assert "--charge Q" in out and "--config C" in out


def _oracle(Z, method, config=None, max_vcycles=100, grid=SMALL):
    if config is None:
        return O.scf(Z, grid["levels"], grid["mixing"], grid["max_r"], grid["delta"], method, max_vcycles=max_vcycles)
    return OC.scf_config(Z, grid["levels"], grid["mixing"], grid["max_r"], grid["delta"], method, config, max_vcycles=max_vcycles)


@pytest.mark.parametrize("method", [0, 1, 2, 3])
def test_oracle_config_with_the_aufbau_is_orc_scf_bit_for_bit(method):
    for Z in (1, 3, 8):
        ref = _oracle(Z, method)
        got = _oracle(Z, method, config=_as4(D.config_aufbau(Z, method)))
        assert got["steps"] == ref["steps"], (Z, method)
        assert got["sorted"] == ref["sorted"] and got["n_steps"] == ref["n_steps"] and got["finished"] == ref["finished"]


# Janak's theorem dE/dn_i = eps_i on the oracle, small-atom grid (LDA), central difference with h = 0.01.  Measured |dE/dn - eps|:
# C 2p at occupation 2: 3.1e-6 Ha (1.1e-5 at h = 0.02, 1.3e-6 at h = 0.005: the O(h^2) error of the difference over a ~7e-7 floor);
# Na 3s at occupation 1: 1.0e-5 Ha (1.3e-5 at h = 0.02, 9.6e-6 at h = 0.005: the discretisation's floor at this grid).  Tolerance:
# 3x the larger figure.
JANAK_H = 0.01
JANAK_TOL = 3e-5
JANAK_CASES = [                     # name, Z, configuration as a function of the occupation x, index of the varied level, x
    ("C 2p", 6, lambda x: [(1, 0, 0, 2.0), (2, 0, 0, 2.0), (2, 1, 0, x)], 2, 2.0),
    ("Na 3s", 11, lambda x: [(1, 0, 0, 2.0), (2, 0, 0, 2.0), (2, 1, 0, 6.0), (3, 0, 0, x)], 3, 1.0),
]


@pytest.mark.parametrize("case", JANAK_CASES, ids=[c[0] for c in JANAK_CASES])
def test_oracle_janak_theorem(case):
    _, Z, cfg, k, x = case
    hi, lo, mid = (_oracle(Z, 0, cfg(x + JANAK_H)), _oracle(Z, 0, cfg(x - JANAK_H)), _oracle(Z, 0, cfg(x)))
    assert hi["finished"] and lo["finished"] and mid["finished"]
    dE = (hi["steps"][-1]["Etotal"] - lo["steps"][-1]["Etotal"]) / (2 * JANAK_H)
    assert abs(dE - mid["steps"][-1]["E"][0][k]) < JANAK_TOL, (dE, mid["steps"][-1]["E"][0][k])


def test_oracle_rejects_malformed_configurations():
    with pytest.raises(ValueError):
        _oracle(6, 0, config=[(1, 0, 1, 2.0)])          # a beta entry in LDA
    with pytest.raises(ValueError):
        _oracle(6, 0, config=[(2, 2, 0, 2.0)])          # l >= n


def _sharded_worker(rank, world, port, ret):
    import sys
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    from dftatom_b200.distributed import solve_sharded
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    opts = [D.Options(3, 9, 12.0, 0.008, 0.5, 0, charge=1), D.Options(4, 9, 12.0, 0.008, 0.5, 0), D.Options(8, 9, 12.0, 0.008, 0.5, 1, charge=-1),
            D.Options(10, 9, 12.0, 0.008, 0.5, 0, config="[He] 2s2 2p5 3s1"), D.Options(6, 9, 12.0, 0.008, 0.5, 0, config="[He] 2s2 2p1.5"),
            D.Options(2, 9, 12.0, 0.008, 0.5, 0)]

    def solve(shard):   # the Options carry their configuration to the rank that solves them
        return [(OC.scf_config(o.Z, o.MultigridLevels, o.alpha, o.MaxR, o.deltaGrid, o.method, o.entries(), max_vcycles=10) if o.configured else
                 O.scf(o.Z, o.MultigridLevels, o.alpha, o.MaxR, o.deltaGrid, o.method, max_vcycles=10))["steps"][-1]["Etotal"] for o in shard]

    res = solve_sharded(opts, solve, rank, world)
    if rank == 0:
        ret["sharded"] = res
        ret["serial"] = solve(opts)
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_of_configured_atoms():
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 31500 + os.getpid() % 2000
    mp.spawn(_sharded_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret["sharded"] == ret["serial"] and len(ret["sharded"]) == 6
