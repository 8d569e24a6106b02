#!/bin/bash
# Per-kernel SASS comparison of two builds of a library (e.g. the parent commit's and this tree's libray_b200.so):
#   tools/sass_diff.sh OLD.so NEW.so
# Splits `cuobjdump -sass` by kernel, keeps only the instruction lines (offsets + opcodes), and normalises the per-file
# hash in anonymous-namespace names (it depends on the build path).  Prints the kernels only one side has and every
# kernel present in both whose instructions differ.
set -e
split() {  # $1 library, $2 output directory
  mkdir -p "$2"
  cuobjdump -sass "$1" | sed -E "s/_GLOBAL__N__[0-9a-f]+_[0-9]+_([A-Za-z_]+)_cu_[0-9a-f]+/_GLOBAL__N_\1/g" |
    awk -v d="$2" '/Function : /{f=d"/"$3".sass"} f && /^[[:space:]]+\/\*[0-9a-f]+\*\//{print > f}'
}
tmp=$(mktemp -d)
trap 'rm -rf "$tmp"' EXIT
split "$1" "$tmp/a"
split "$2" "$tmp/b"
echo "kernels: $(ls "$tmp/a" | wc -l) -> $(ls "$tmp/b" | wc -l)"
echo "only in $2:"; comm -13 <(ls "$tmp/a") <(ls "$tmp/b") | sed 's/\.sass$//'
echo "only in $1:"; comm -23 <(ls "$tmp/a") <(ls "$tmp/b") | sed 's/\.sass$//'
nd=0
for f in $(comm -12 <(ls "$tmp/a") <(ls "$tmp/b")); do
  cmp -s "$tmp/a/$f" "$tmp/b/$f" || { echo "DIFFERS: ${f%.sass}"; nd=$((nd + 1)); }
done
echo "kernels in both whose SASS differs: $nd"
