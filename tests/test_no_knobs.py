"""The library has one build and one code path per input: no environment variable or -D override selects or retunes a
computation. Paths are chosen from what the code can observe (batch size, image width, levels, overlapping inputs).
Two environment variables remain: EA_SOLVE_DEBUG only observes (cycle counters), and EA_SHARD_MODE=nccl selects the
host-driven point-sharded path, the one that GPUs without peer access run."""
import os
import re

from conftest import ROOT

CSRC = os.path.join(ROOT, "edge_alignment_b200", "csrc")
ALLOWED_ENV = {"EA_SOLVE_DEBUG", "EA_SHARD_MODE"}


def sources():
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".h", ".cpp")):
            yield f, open(os.path.join(CSRC, f)).read()


def test_only_observing_env_vars():
    seen = set()
    for f, src in sources():
        for m in re.finditer(r"\bgetenv\s*\(\s*(\"([^\"]*)\")?", src):
            assert m.group(1), "%s: getenv without a literal name" % f
            seen.add(m.group(2))
    assert seen == ALLOWED_ENV, "environment variables read by the library: %s" % sorted(seen)


def header_guard(f, directives):
    """The macro of a classic include guard: a header's first directive `#ifndef X` followed by `#define X`."""
    if f.endswith((".h", ".cuh")) and len(directives) >= 2:
        (k0, a0), (k1, a1) = directives[0], directives[1]
        if k0 == "ifndef" and k1 == "define" and a0.split()[:1] == a1.split()[:1]:
            return a0.split()[0]
    return None


def test_no_compile_time_switches():
    for f, src in sources():
        directives = re.findall(r"^[ \t]*#[ \t]*(\w+)[ \t]*(.*)$", src, flags=re.M)
        guard = header_guard(f, directives)
        for i, (kind, arg) in enumerate(directives):
            if kind not in ("if", "ifdef", "ifndef", "elif"):
                continue
            names = set(re.findall(r"\b[A-Za-z_]\w*\b", arg.split("//")[0])) - {"defined", guard}
            keyed = sorted(n for n in names if re.match(r"(EA|VB)_", n))
            assert not keyed, "%s: #%s %s" % (f, kind, arg)
            # an override guard under any name: #ifndef X followed by #define X
            if kind == "ifndef" and i + 1 < len(directives) and directives[i + 1][0] == "define":
                assert directives[i + 1][1].split()[:1] != arg.split()[:1] or arg.split()[0] == guard, \
                    "%s: -D override guard on %s" % (f, arg.split()[0])
