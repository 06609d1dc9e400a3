#!/bin/sh
# sass_diff.sh OLD.so NEW.so [SED_EXPR] — diff the SASS of two builds of librt_b200.so function by function.
#
# Every function of OLD must exist in NEW with identical instructions (addresses and column padding ignored).
# SED_EXPR maps an OLD mangled name to its NEW one where a template gained an argument.  Example: k_extend gained
# the query mode Q and a trailing QueryArgs parameter, so the RENDER instantiations are compared under
#   's/^(_ZN2rt8k_extendILb.ELb.ELb.)EEEvNS_9SceneViewENS_10PathArraysEP6float4PKjPjPy$/\1ELNS_5QueryE0EEEvNS_9SceneViewENS_10PathArraysEP6float4PKjPjPyNS_9QueryArgsE/'
# Prints the functions that differ or are missing (nothing else) and exits 1 if there is any.
set -e
[ $# -ge 2 ] || { echo "usage: $0 OLD.so NEW.so [SED_EXPR]" >&2; exit 2; }
CUOBJDUMP=${CUOBJDUMP:-/usr/local/cuda/bin/cuobjdump}
tmp=$(mktemp -d)
trap 'rm -rf "$tmp"' EXIT
split() {  # $1 = .so, $2 = output directory: one file per function
    mkdir -p "$2"
    "$CUOBJDUMP" -sass "$1" | awk -v d="$2" '
        /Function : / { f = d "/" $3; next }
        /^[ \t]*(Fatbin|identifier|arch|code version|host|compile_size)/ { f = ""; next }
        f { line = $0; sub(/\/\*[0-9a-f]+\*\//, "", line); gsub(/[ \t]+/, " ", line); print line > f }'
}
split "$1" "$tmp/old"
split "$2" "$tmp/new"
bad=0
for p in "$tmp"/old/*; do
    f=$(basename "$p")
    g=$f
    [ $# -ge 3 ] && g=$(echo "$f" | sed -E "$3")
    if [ ! -f "$tmp/new/$g" ]; then echo "missing in NEW: $f"; bad=1
    elif ! cmp -s "$p" "$tmp/new/$g"; then echo "differs: $f"; bad=1
    fi
done
exit $bad
