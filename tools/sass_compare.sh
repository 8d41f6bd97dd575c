#!/bin/bash
# CPU-only check that a refactor of the CUDA sources leaves the machine code alone. Builds the default FORMATS of
# BASE_REV (git archive into a temporary directory) and of the working tree with -Xptxas -v, splits `cuobjdump -sass`
# of every object per function and compares the two builds function by function, then diffs the -Xptxas -v output
# (registers, stack frame, shared memory, spills) of every object.
# usage: tools/sass_compare.sh BASE_REV [SED_EXPR]
#   SED_EXPR maps the base build's demangled function names onto the working tree's, for a kernel renamed on purpose,
#   e.g.  tools/sass_compare.sh main 's/render_rc_kernel<5, /render_rc_kernel</'
# Exit status 0 when every function of BASE_REV is present and identical and the ptxas output matches.
set -euo pipefail
BASE=${1:?usage: tools/sass_compare.sh BASE_REV [SED_EXPR]}; MAP=${2:-}
ROOT=$(git rev-parse --show-toplevel)
TMP=$(mktemp -d); trap 'rm -rf "$TMP"' EXIT
mkdir -p "$TMP/src"
git -C "$ROOT" archive "$BASE" spectroplot-js_b200/csrc include | tar -x -C "$TMP/src"
# one ptxas log per object: parallel jobs would interleave their stderr
printf '#!/bin/sh\nfor a; do [ "$p" = -o ] && o=$a; p=$a; done\nexec %s "$@" 2> "$o.log"\n' "$(command -v "${NVCC:-nvcc}")" > "$TMP/nvcc"
chmod +x "$TMP/nvcc"

# names of file-local functions carry a hash of the source: drop it; then apply the rename map
norm() { sed -E -e 's/_INTERNAL_[0-9a-f]+_/_INTERNAL_/g' -e "${1:-}"; }

# build SRC_ROOT NAME SED_EXPR: objects and logs in $TMP/NAME, one SASS file per function in $TMP/NAME.sass/<object>/,
# "<object> <demangled name> <file>" lines in $TMP/NAME.names
build() {
    make -s -j "$(nproc)" -C "$1/spectroplot-js_b200/csrc" NVCC="$TMP/nvcc" OUT="$TMP/$2" OBJ="$TMP/$2" XFLAGS="-Xptxas -v" >&2 || { cat "$TMP/$2"/*.log >&2; exit 1; }
    for o in "$TMP/$2"/*.o; do
        obj=$(basename "$o" .o); mkdir -p "$TMP/$2.sass/$obj"
        cuobjdump -sass "$o" | awk -v dir="$TMP/$2.sass/$obj" '/Function : / { f = dir "/" ++n; print $3; next } f { print > f }' \
          | c++filt | norm "${3:-}" | awk -v obj="$obj" '{ print obj " " $0 "\t" obj "/" NR }'
        grep -v "Compile time" "$o.log" | c++filt | norm "${3:-}" > "$TMP/$2.sass/$obj.ptxas"
    done | sort > "$TMP/$2.names"
}
build "$TMP/src" base "$MAP"
build "$ROOT" new ""

nfun=0; nbad=0
while IFS=$'\t' read -r key f; do
    nfun=$((nfun + 1))
    g=$(awk -F'\t' -v k="$key" '$1 == k { print $2 }' "$TMP/new.names")
    if [ -z "$g" ]; then echo "missing in the working tree: $key"; nbad=$((nbad + 1))
    elif ! cmp -s "$TMP/base.sass/$f" "$TMP/new.sass/$g"; then echo "differs: $key"; nbad=$((nbad + 1)); fi
done < "$TMP/base.names"
echo "$nfun functions in $BASE, $(wc -l < "$TMP/new.names") in the working tree: $nbad missing or different"
for p in "$TMP"/base.sass/*.ptxas; do
    if ! diff "$p" "$TMP/new.sass/$(basename "$p")"; then echo "ptxas -v differs: $(basename "$p" .ptxas)"; nbad=$((nbad + 1)); fi
done
[ "$nbad" -eq 0 ] && echo "identical, ptxas -v output included"
