"""Per-function SASS comparison of two builds: proves that a change left kernels measured on hardware untouched.

    python scripts/sass_diff.py snapshot DIR          # cuobjdump -sass of every aecf_b200/csrc/build/*.o into DIR
    python scripts/sass_diff.py compare BEFORE AFTER   # functions whose instruction stream differs, added, removed
    python scripts/sass_diff.py compare BEFORE AFTER --pair ARG
                                                       # the same, after a new trailing template argument: an old function
                                                       # is compared with the new one whose last template argument is ARG
                                                       # (ARG "=": the one whose last argument repeats the one before it,
                                                       # f<float> -> f<float, float> and f<bf16> -> f<bf16, bf16> at once)
    python scripts/sass_diff.py manifest DIR OUT.json  # {demangled function: [sha1, instructions]} of a snapshot
    python scripts/sass_diff.py check OUT.json DIR     # a snapshot against a committed manifest (exit 1 on a change)

Instruction text only (addresses, encodings and comments are dropped), keyed by mangled function name.
"""
import glob
import hashlib
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "aecf_b200", "csrc", "build")


def snapshot(dest):
    os.makedirs(dest, exist_ok=True)
    for obj in sorted(glob.glob(os.path.join(BUILD, "*.o"))):
        out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
        with open(os.path.join(dest, os.path.basename(obj)[:-2] + ".sass"), "w") as f:
            f.write(out)


INSTR = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*/\*")


def functions(path):
    """{mangled name: (sha1 of the instruction text, instruction count)}"""
    table, name, h, n = {}, None, None, 0
    for line in open(path):
        if "Function :" in line:
            if name is not None:
                table[name] = (h.hexdigest(), n)
            name, h, n = line.split("Function :")[1].strip(), hashlib.sha1(), 0
            continue
        m = INSTR.match(line)
        if m and name is not None:
            h.update(m.group(1).encode())
            n += 1
    if name is not None:
        table[name] = (h.hexdigest(), n)
    return table


def load(directory):
    table = {}
    for path in sorted(glob.glob(os.path.join(directory, "*.sass"))):
        table.update(functions(path))
    return table


def paired(a, b, arg):
    """Rename the functions of `b` whose last template argument is `arg` to the name they had without it (when `a` has
    that name), e.g. f<float, 3, false> -> f<float, 3> for arg = "false"."""
    names = demangle_all(sorted(b))
    old = {v: k for k, v in demangle_all(sorted(a)).items()}
    out, pairs = {}, 0
    for k, v in b.items():
        if arg == "=":
            head, sep, tail = names[k].rpartition(">(")
            pre, comma, last = head.rpartition(", ")
            sep = sep if comma and re.split(r"<|, ", pre)[-1] == last else ""
            head = pre
        else:
            head, sep, tail = names[k].rpartition(f", {arg}>(")
        key = old.get(head + ">(" + tail) if sep else None
        if key is not None:
            out[key] = v
            pairs += 1
        else:
            out[k] = v
    what = "a repeated" if arg == "=" else "the"
    print(f"{pairs} functions paired with their name before {what} trailing template argument" + ("" if arg == "=" else f" {arg}"))
    return out


def compare(before, after, pair=None):
    a, b = load(before), load(after)
    if pair is not None:
        b = paired(a, b, pair)
    changed = sorted(k for k in a if k in b and a[k] != b[k])
    removed = sorted(k for k in a if k not in b)
    added = sorted(k for k in b if k not in a)
    print(f"{len(a)} functions before, {len(b)} after: {len(changed)} changed, {len(removed)} removed, {len(added)} added")
    for title, names in (("changed", changed), ("removed", removed), ("added", added)):
        for k in names[:40]:
            demangled = subprocess.run(["c++filt", k], capture_output=True, text=True).stdout.strip()[:150]
            extra = f"  {a[k][1]} -> {b[k][1]} instructions" if title == "changed" else ""
            print(f"  {title}: {demangled}{extra}")
        if len(names) > 40:
            print(f"  ... and {len(names) - 40} more {title}")
    return 1 if (changed or removed) else 0


def demangle_all(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    return dict(zip(names, out))


def manifest(directory, out_path):
    import json
    table = load(directory)
    names = demangle_all(sorted(table))
    with open(out_path, "w") as f:
        json.dump({names[k]: list(v) for k, v in sorted(table.items())}, f, indent=0, sort_keys=True)
    print(f"{len(table)} functions -> {out_path}")


def check(manifest_path, directory):
    import json
    want = json.load(open(manifest_path))
    table = load(directory)
    names = demangle_all(sorted(table))
    got = {names[k]: list(v) for k, v in table.items()}
    changed = sorted(k for k in want if k in got and got[k] != want[k])
    removed = sorted(k for k in want if k not in got)
    added = sorted(k for k in got if k not in want)
    print(f"{len(want)} functions in the manifest, {len(got)} in the build: {len(changed)} changed, {len(removed)} removed, {len(added)} added")
    for title, group in (("changed", changed), ("removed", removed), ("added", added)):
        for k in group[:40]:
            print(f"  {title}: {k[:150]}")
    return 1 if (changed or removed) else 0


if __name__ == "__main__":
    if len(sys.argv) >= 3 and sys.argv[1] == "snapshot":
        snapshot(sys.argv[2])
    elif len(sys.argv) >= 4 and sys.argv[1] == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3], sys.argv[5] if len(sys.argv) >= 6 and sys.argv[4] == "--pair" else None))
    elif len(sys.argv) >= 4 and sys.argv[1] == "manifest":
        manifest(sys.argv[2], sys.argv[3])
    elif len(sys.argv) >= 4 and sys.argv[1] == "check":
        sys.exit(check(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
