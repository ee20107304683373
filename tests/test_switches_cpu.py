"""Every environment variable the library and the package read is documented in DESIGN.md section 8 ("Developer
switches"), and the table lists nothing that is no longer read (no GPU needed)."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "super_resolution-image-reconstructer-multi_generator_gan_b200")
READS = re.compile(r'(?:getenv\(|os\.environ\.get\(|os\.environ\[)\s*"(SRG_\w+)"')


def read_switches():
    files = glob.glob(os.path.join(PKG, "csrc", "*.cu")) + glob.glob(os.path.join(PKG, "csrc", "*.cuh")) + \
        glob.glob(os.path.join(PKG, "*.py"))
    names = set()
    for f in files:
        with open(f) as fh:
            names |= set(READS.findall(fh.read()))
    return names


def documented_switches():
    with open(os.path.join(ROOT, "DESIGN.md")) as fh:
        text = fh.read()
    section = text[text.index("### Developer switches"):]
    section = section[:section.index("\n## ")]
    rows = [line for line in section.splitlines() if line.startswith("| `")]
    return {n for row in rows for n in re.findall(r"SRG_\w+", row.split("|")[1])}


def test_every_switch_read_is_documented_and_every_documented_switch_is_read():
    read, documented = read_switches(), documented_switches()
    assert read == documented, {"read but not in DESIGN.md section 8": sorted(read - documented),
                                "in DESIGN.md section 8 but not read": sorted(documented - read)}
