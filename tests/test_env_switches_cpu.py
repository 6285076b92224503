"""Every environment variable the package reads is documented: the `B200PPO_*` string literals in the CUDA sources and
the package's Python files are exactly the names in the "Environment variables" table of profiles/README.md."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "mujoco_reinforcement_learning_b200")
# a quoted name, wherever it stands: getenv("X"), getenv(a ? "X" : "Y"), os.environ.get("X", ...)
LITERAL = re.compile(r"""["'](B200PPO_[A-Z0-9_]+)["']""")


def _names_in_code():
    files = sorted(glob.glob(os.path.join(PKG, "csrc", "*")) + glob.glob(os.path.join(PKG, "*.py")))
    names = {}
    for path in files:
        for name in LITERAL.findall(open(path, encoding="utf-8").read()):
            names.setdefault(name, os.path.relpath(path, ROOT))
    return names


def _names_in_table():
    text = open(os.path.join(ROOT, "profiles", "README.md"), encoding="utf-8").read()
    section = text.split("\n## Environment variables\n", 1)
    assert len(section) == 2, "profiles/README.md has no '## Environment variables' section"
    body = section[1].split("\n## ", 1)[0]
    return set(re.findall(r"^\| `(B200PPO_[A-Z0-9_]+)` \|", body, flags=re.M))


def test_scan_sees_every_literal_form():
    src = 'getenv(w ? "B200PPO_A_WGRAD" : "B200PPO_A"); os.environ.get(\'B200PPO_B\', "1")'
    assert LITERAL.findall(src) == ["B200PPO_A_WGRAD", "B200PPO_A", "B200PPO_B"]


def test_every_env_switch_is_documented():
    code = _names_in_code()
    table = _names_in_table()
    assert code, "no B200PPO_* names found in the sources"
    undocumented = sorted(f"{n} ({code[n]})" for n in set(code) - table)
    stale = sorted(table - set(code))
    assert not undocumented, f"read but missing from the profiles/README.md table: {undocumented}"
    assert not stale, f"in the profiles/README.md table but read nowhere: {stale}"
