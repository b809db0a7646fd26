"""CPU: every LLAMAX_* environment variable the package reads is a row of README's switch table, and every LLAMAX_* row
of that table is read by the package. A switch that changes what runs has to be documented on purpose."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "llamax_b200")

# os.environ.get("X") / os.environ["X"] / os.getenv("X") in Python, getenv("X") in the CUDA sources
_READ = re.compile(r"""(?:environ\.get\(|environ\[|getenv\()\s*["'](LLAMAX_\w+)["']""")


def _switches_read() -> set:
    names = set()
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                with open(os.path.join(dirpath, f), encoding="utf-8") as fh:
                    names.update(_READ.findall(fh.read()))
    return names


def _switches_documented() -> set:
    with open(os.path.join(ROOT, "README.md"), encoding="utf-8") as fh:
        text = fh.read()
    section = text.split("\n## Environment switches\n", 1)[1].split("\n## ", 1)[0]
    names = set()
    for line in section.splitlines():
        if line.startswith("|"):
            names.update(re.findall(r"`(LLAMAX_\w+)`", line.split("|")[1]))
    return names


def test_every_switch_read_is_documented_and_every_documented_switch_is_read():
    read, documented = _switches_read(), _switches_documented()
    assert read == documented, (f"read but not in README's switch table: {sorted(read - documented)}; "
                                f"in the table but never read: {sorted(documented - read)}")
