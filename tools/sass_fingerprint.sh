#!/bin/bash
# One md5 per kernel of the library's SASS: encodings stripped and the offsets of constant-bank 0
# (kernel parameters) masked, so a kernel whose parameter struct lost a field still matches when
# its instruction stream is unchanged.  Two builds with the same line for a kernel run the same
# device code for it; a kernel added or removed elsewhere in the same object does not show up in
# the others' hashes.   usage: tools/sass_fingerprint.sh [csrc dir]
# output lines: <object> <hash> <mangled kernel name>, sorted; the hashes in the names of anonymous
# namespaces (they depend on the checkout's path) are masked so that listings of two checkouts line up
d=${1:-diskann_b200/csrc}
for o in "$d"/*.o; do
  cuobjdump -sass "$o" | python3 -c '
import hashlib, re, sys
obj, fn, body = sys.argv[1], None, []
def emit():
    if fn: print(obj, hashlib.md5("".join(body).encode()).hexdigest()[:16], fn)
for line in sys.stdin:
    m = re.match(r"\s+Function : (\S+)", line)
    if m:
        emit()
        fn, body = re.sub(r"_GLOBAL__N__[0-9a-f]{8}_(\d+_\w+?_cu_)[0-9a-f]{8}", r"_GLOBAL__N__*_\1*", m.group(1)), []
    elif re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
        line = re.sub(r"/\* 0x[0-9a-f]* \*/", "", line)
        body.append(re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][*]", line))
emit()
' "$(basename "$o" .o)"
done | sort
