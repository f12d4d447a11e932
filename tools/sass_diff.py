"""Compare the SASS of every kernel of one build of libcpflow_b200.so with another build.

    python tools/sass_diff.py OLD.so NEW.so

Prints, per kernel symbol of OLD, whether NEW has it with identical SASS (`cuobjdump -sass`), and the symbols NEW adds.
Exit status 1 when a kernel of OLD is missing from NEW or differs: a change that must leave existing kernels alone
(new instantiations only) is checked this way without a GPU.
"""
import re
import shutil
import subprocess
import sys


def _cuobjdump():
    for c in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if c:
            return c
    raise SystemExit("cuobjdump not found")


def sass_by_function(lib):
    out = subprocess.run([_cuobjdump(), "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = "\n".join(body)
            # anonymous namespaces are mangled with a hash of their translation unit: compare by the rest of the name
            name, body = re.sub(r"_GLOBAL__N__[0-9A-Za-z_]+?_(?=\d)", "_GLOBAL__N_", m.group(1)), []
        elif name and "/*" in line:          # instructions and their encodings, not the cubin headers in between
            body.append(line.rstrip())
    if name:
        funcs[name] = "\n".join(body)
    return funcs


def main(old_lib, new_lib):
    old, new = sass_by_function(old_lib), sass_by_function(new_lib)
    same = sum(1 for k in old if new.get(k) == old[k])
    changed = [k for k in old if k in new and new[k] != old[k]]
    missing = [k for k in old if k not in new]
    added = sorted(k for k in new if k not in old)
    for k in changed:
        print("DIFFERS ", k)
    for k in missing:
        print("MISSING ", k)
    for k in added:
        print("added   ", k)
    print(f"{len(old)} kernels in {old_lib}: {same} identical, {len(changed)} differ, {len(missing)} missing; "
          f"{len(added)} added in {new_lib}")
    return 1 if changed or missing else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        raise SystemExit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
