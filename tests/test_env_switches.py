"""The environment variables the library reads, host-only.  Kernel selection follows the shapes; an environment switch
is a second code path that no test exercises, so each one the library reads is a deliberate decision listed here."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "glfusion_b200")

KEPT = {
    "GLF_DOT_ALGO",        # bench.py reads it for the algorithm threshold
    "GLF_GRAM_CHAIN",      # bench.py reads it for the launch count
    "GLF_P2P_TIMEOUT_S",   # bounds the peer wait of the all-reduce
    "GLF_CHAIN_TRACE",     # clock-trace instrumentation: never changes which code computes a result
    "GLF_GRAM_TRACE",
    "GLF_WGRAD_TRACE",
}

_C_GETENV = re.compile(r"\bgetenv\s*\(\s*\"(\w+)\"")
_PY_ENV = re.compile(r"\bos\.(?:environ(?:\s*\.\s*\w+\s*\(|\s*\[)|getenv\s*\()\s*[\"'](GLF_\w+)[\"']")


def _read_all(top, exts):
    for d, _, files in os.walk(top):
        for f in files:
            if f.endswith(exts):
                with open(os.path.join(d, f), encoding="utf-8") as fh:
                    yield fh.read()


def test_environment_switches_are_the_kept_list():
    names = set()
    for src in _read_all(os.path.join(PKG, "csrc"), (".cu", ".cuh", ".h", ".cpp")):
        names.update(n for n in _C_GETENV.findall(src) if n.startswith("GLF_"))
    for src in _read_all(PKG, (".py",)):
        names.update(_PY_ENV.findall(src))
    assert names == KEPT, f"unexpected: {sorted(names - KEPT)}, missing: {sorted(KEPT - names)}"
