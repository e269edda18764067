"""Per-kernel SASS digests of libessentials_b200.so, to show that a refactor left the machine code alone:
    python scripts/sass_digest.py OLD.so NEW.so    (or one .so to print its digests)
Each `Function :` block is hashed with its /*addr*/ prefixes stripped; the per-build hashes in internal names
depend on the source path and are normalised. Exits 1 when the kernel sets or any digest differ."""
import hashlib
import re
import subprocess
import sys

HASHED = re.compile(r"_INTERNAL_[0-9a-f]{8}_|_GLOBAL__N__[0-9a-f]{8}_")


def digests(so):
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    out, name, body = {}, None, []
    for line in sass.splitlines() + ["Function : end"]:
        m = re.match(r"\s*Function : (.*)", line)
        if m:
            if name is not None:  # a kernel instantiated in several translation units has one copy in each
                out.setdefault(name, []).append(hashlib.sha256("\n".join(body).encode()).hexdigest()[:16])
            name, body = HASHED.sub("_H_", m.group(1).strip()), []
        elif name is not None and "/*" in line:
            body.append(HASHED.sub("_H_", re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)).strip())
    return {k: ",".join(sorted(v)) for k, v in out.items()}


if len(sys.argv) == 2:
    for name, d in sorted(digests(sys.argv[1]).items()):
        print(d, name)
    sys.exit(0)
old, new = digests(sys.argv[1]), digests(sys.argv[2])
gone, added = sorted(old.keys() - new.keys()), sorted(new.keys() - old.keys())
changed = sorted(k for k in old.keys() & new.keys() if old[k] != new[k])
for tag, names in (("only in old", gone), ("only in new", added), ("SASS differs", changed)):
    for k in names:
        print(f"{tag}: {k}")
print(f"{len(old)} old, {len(new)} new kernels; {len(changed)} differ, {len(gone)} gone, {len(added)} added")
sys.exit(1 if gone or added or changed else 0)
