"""Text report in the reference's format, and its parser.

The reference's only result channel is text on std::cout (DFTAtom.cpp:358,398,548-556,472,476,483,
487-490; LSDA :857,1015-1021).  `format_report` reproduces those lines from per-step records so the
headless CLI's output can be diffed against the reference's; `parse_report` turns either program's
stdout back into records (used by the golden generator and the parity tests).
"""
import re

ORB = "spdf"
SEP = "*" * 80

_E_RE = re.compile(r"^Energy (?:alpha |beta )?(\d+)([spdf]): (\S+) Num nodes: (-?\d+)$")
_T_RE = re.compile(r"^Etotal = (\S+) Ekin = (\S+) Ecoul = (\S+) Eenuc = (\S+) Exc = (\S+)$")
_H_RE = re.compile(r"^Computing atom with Z=(\d+) using (LSDA|LSD|LDA) with (non-uniform|uniform) grid$")
_C_RE = re.compile(r"(\d+)([spdf])(\d+)")


def parse_report(text):
    """Parse reference-format stdout into {Z, method, steps:[{levels:[{n,l,E,nodes}], Etotal,...}], finished, final}."""
    rec = dict(Z=None, method=None, steps=[], finished=False, final=None)
    cur = None
    for line in text.splitlines():
        line = line.rstrip()
        m = _H_RE.match(line)
        if m:
            rec["Z"] = int(m.group(1))
            rec["method"] = 1 if m.group(2) == "LSDA" else 0
            rec["grid"] = m.group(3)          # "uniform": the CalculateUniform* pair (DFTAtom.cpp:69, :655), levels tagged alpha / beta
            continue
        if line.startswith("Step: "):
            cur = dict(step=int(line[6:]), levels=[])
            rec["steps"].append(cur)
            continue
        m = _E_RE.match(line)
        if m and cur is not None:
            cur["levels"].append(dict(n=int(m.group(1)), l=ORB.index(m.group(2)), E=float(m.group(3)), nodes=int(m.group(4))))
            continue
        m = _T_RE.match(line)
        if m and cur is not None:
            for k, v in zip(("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc"), m.groups()):
                cur[k] = float(v)
            continue
        if line == "Finished!":
            rec["finished"] = True
            continue
        if line.startswith("Alpha: "):
            rec["final"] = dict(alpha=[(int(a), ORB.index(b), int(c)) for a, b, c in _C_RE.findall(line[7:])])
            continue
        if line.startswith("Beta: ") and rec["final"] is not None:
            rec["final"]["beta"] = [(int(a), ORB.index(b), int(c)) for a, b, c in _C_RE.findall(line[6:])]
            continue
        if rec["steps"] and _C_RE.match(line) and rec["final"] is None:
            rec["final"] = dict(alpha=[(int(a), ORB.index(b), int(c)) for a, b, c in _C_RE.findall(line)])
    return rec


def _fmt(x, precision):
    return f"{x:.{precision}f}" if precision <= 6 else f"{x:.{precision}g}"


def format_report(Z, method, steps, finished, final_alpha, final_beta=None, precision=6, n_alpha=None):
    """Inverse of parse_report: the exact line sequence the reference prints (DFTAtom.cpp:358-490 / :857-1021).

    steps: list of dicts {levels: [(n, l, E, nodes), ...] (alpha first, then beta, untagged as in the reference's
    non-uniform path), Etotal, Ekin, Ecoul, Eenuc, Exc}; final_*: [(n, l, occ), ...] sorted by eigenvalue.
    """
    # method 2 / 3: the uniform-grid pair (DFTAtom.cpp:69 "LDA", :656 "LSDA"; its LSDA level lines are tagged alpha / beta, :269-277)
    uniform = method >= 2
    lsda = method in (1, 3)
    out = [f"Computing atom with Z={Z} using {('LSDA' if lsda else ('LDA' if uniform else 'LSD'))} with {'uniform' if uniform else 'non-uniform'} grid"]
    for k, st in enumerate(steps):
        out.append(f"Step: {k}")
        for j, (n, l, E, nodes) in enumerate(st["levels"]):
            tag = ""
            if uniform and lsda:
                tag = "alpha " if (n_alpha is None or j < n_alpha) else "beta "
            out.append(f"Energy {tag}{n}{ORB[l]}: {_fmt(E, precision)} Num nodes: {nodes}")
        out.append("Etotal = {} Ekin = {} Ecoul = {} Eenuc = {} Exc = {}".format(
            *[_fmt(st[key], precision) for key in ("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc")]))
        if finished and k == len(steps) - 1:
            out += ["", "Finished!", ""]
        else:
            out.append(SEP)
    conf = lambda lv: "".join(f"{n}{ORB[l]}{occ:g} " for (n, l, occ) in lv)      # %g: integers as the reference prints them
    if lsda:
        out.append("Alpha: " + conf(final_alpha))
        out.append("Beta: " + conf(final_beta or []))
    else:
        out.append(conf(final_alpha))
    return "\n".join(out) + "\n"
