r"""Compare the SASS of two builds of a library kernel by kernel (cuobjdump -sass; no GPU needed).

    python tools/sass_diff.py OLD.so NEW.so [--rename PATTERN REPLACEMENT]

Prints, per kernel, whether its instructions are identical (encodings and offsets included), and lists the kernels
only one side has. Exit code 1 when a kernel both sides have differs. --rename applies re.sub(PATTERN, REPLACEMENT) to
OLD's kernel names first, for a kernel whose mangled name gained a template argument (e.g. 'ELi(\d)EEEv' ->
'ELi\1ELi0EEEv' for an added trailing int parameter)."""
from __future__ import annotations

import re
import subprocess
import sys


def kernels(path: str, cuobjdump: str = 'cuobjdump') -> dict:
    out = subprocess.run([cuobjdump, '-sass', path], check=True, stdout=subprocess.PIPE, text=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            if name is not None:
                funcs[name] = body
            name, body = m.group(1), []
        elif name is not None and line.strip().startswith('/*'):
            body.append(line.strip())
    if name is not None:
        funcs[name] = body
    return funcs


def main(argv) -> int:
    old, new = kernels(argv[0]), kernels(argv[1])
    if len(argv) == 5 and argv[2] == '--rename':
        old = {re.sub(argv[3], argv[4], k): v for k, v in old.items()}
    elif len(argv) != 2:
        sys.exit(__doc__)
    same = sorted(k for k in old if k in new and old[k] == new[k])
    changed = sorted(k for k in old if k in new and old[k] != new[k])
    removed = sorted(k for k in old if k not in new)
    added = sorted(k for k in new if k not in old)
    print(f"kernels: {len(old)} before, {len(new)} after; {len(same)} instruction-identical, {len(changed)} changed, "
          f"{len(removed)} removed, {len(added)} added")
    for k in changed:
        print(f"  changed: {k} ({len(old[k])} -> {len(new[k])} lines)")
    for k in removed:
        print(f"  removed: {k}")
    for k in added:
        print(f"  added:   {k} ({len(new[k])} lines)")
    return 1 if changed or removed else 0


if __name__ == '__main__':
    sys.exit(main(sys.argv[1:]))
