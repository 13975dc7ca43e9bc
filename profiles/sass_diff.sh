#!/bin/bash
# Per-kernel SASS comparison of two builds of one .cu file: prints SAME / DIFF / MISSING per kernel of the first object.
# Mangled-name parts that only a template parameter added (the PE = false argument and the coupling-plane parameters of
# the Potts kernels) are stripped before matching, and instruction addresses are ignored.
# Usage: profiles/sass_diff.sh old.o new.o
set -e
dump() { cuobjdump -sass "$1" | sed -E 's@/\*[0-9a-f]{4,}\*/@@; s/[[:space:]]+$//'; }
split() { awk -v dir="$2" '/Function : /{name=$3; gsub(/Lb0E/,"",name); gsub(/PKS2_S4_/,"",name); f=dir"/"name".sass"} f{print > f}' <(dump "$1"); }
tmp=$(mktemp -d)
trap 'rm -rf "$tmp"' EXIT
mkdir "$tmp/a" "$tmp/b"
split "$1" "$tmp/a"
split "$2" "$tmp/b"
for f in "$tmp"/a/*.sass; do
    n=$(basename "$f" .sass)
    if [ ! -f "$tmp/b/$n.sass" ]; then echo "MISSING $n"; continue; fi
    if diff <(tail -n +2 "$f") <(tail -n +2 "$tmp/b/$n.sass") >/dev/null; then echo "SAME    $n"; else echo "DIFF    $n"; fi
done
