#!/usr/bin/env bash
# TEST INFRASTRUCTURE. Builds the reference's own C++ (the original SCSsim
# sources, read at BASELINE.json's reference_path, or where $SCS_REFERENCE_DIR
# points when it is set) into oracle/_ref/ — two binaries:
#   oracle/_ref/bin/scssim         the reference + the five missing `return`s
#                                  (SURVEY.md §8c: without them g++ >= 8 emits
#                                  code that crashes); behaviour otherwise stock.
#   oracle/_ref/bin/scssim_replay  same + seed from $SCS_SEED and a log of every
#                                  random draw to $SCS_REPLAY_LOG.* (ref_hooks.h).
# Nothing from the reference is committed: the patched copies live only under
# the git-ignored oracle/_ref/src. Uses g++ directly (no cmake).
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
REF="${SCS_REFERENCE_DIR-$(python3 -c 'import json, sys; print(json.load(open(sys.argv[1])).get("reference_path", ""))' "$HERE/../BASELINE.json")}"
OUT="$HERE/_ref"
if [ -z "$REF" ] || [ ! -d "$REF/lib" ]; then
    if [ -x "$OUT/bin/scssim" ] && [ -x "$OUT/bin/scssim_replay" ]; then
        echo "build_ref: no SCSsim sources at '$REF', keeping prebuilt $OUT/bin" >&2; exit 0
    fi
    echo "build_ref: no SCSsim sources at '$REF' and no prebuilt binaries" >&2; exit 1
fi
if [ -x "$OUT/bin/scssim" ] && [ -x "$OUT/bin/scssim_replay" ] && \
   [ "$OUT/bin/scssim_replay" -nt "$HERE/ref_hooks.cpp" ] && [ "$OUT/bin/scssim_replay" -nt "$HERE/build_ref.sh" ]; then
    exit 0
fi
rm -rf "$OUT/src" "$OUT/src_replay"; mkdir -p "$OUT/src" "$OUT/src_replay" "$OUT/bin"

MODS="amplicon config fastahack fragment genome malbac matrix mydefine profile psifunc seqwriter snp split threadpool vcfparser"
for d in $MODS; do cp -r "$REF/lib/$d" "$OUT/src/$d"; done
cp "$REF/src/scssim.cpp" "$OUT/src/scssim.cpp"

# expect LINE FILE REGEX : fail loudly if the reference is not the revision the patch was written for
expect() { sed -n "$1p" "$2" | grep -Eq "$3" || { echo "build_ref: $2:$1 does not match /$3/" >&2; exit 1; }; }

S="$OUT/src"
# --- patch 1: the five missing returns (applied to both variants) -----------
expect 151 "$S/fragment/Fragment.cpp" 'extendSemiAmplicons\(results\)'
sed -i '151a\	return NULL;' "$S/fragment/Fragment.cpp"
expect 393 "$S/amplicon/Amplicon.cpp" '^\s*}\s*$'
sed -i '393a\	return NULL;' "$S/amplicon/Amplicon.cpp"
expect 252 "$S/amplicon/Amplicon.cpp" 'extendFullAmplicons\(results\)'
sed -i '252a\	return NULL;' "$S/amplicon/Amplicon.cpp"
expect 271 "$S/mydefine/MyDefine.cpp" '^\s*}\s*$'
sed -i '271a\	return ret;' "$S/mydefine/MyDefine.cpp"
expect 200 "$S/mydefine/MyDefine.cpp" '^\s*}\s*$'
sed -i '200a\	return NULL;' "$S/mydefine/MyDefine.cpp"

cp -r "$S/." "$OUT/src_replay/"
R="$OUT/src_replay"
# --- patch 2 (replay variant only): seeds + draw log ------------------------
expect 47 "$R/scssim.cpp" 'srand\(start_t\)'
sed -i '47s/srand(start_t)/srand(scs_ref_seed(0, (unsigned) start_t))/' "$R/scssim.cpp"
expect 41 "$R/threadpool/ThreadPool.cpp" 'unsigned seed = chrono'
sed -i '41a\		seed = scs_ref_seed(1000 + (unsigned) i, seed);' "$R/threadpool/ThreadPool.cpp"
# (line numbers below are +1 in ThreadPool.cpp because of the insertion above)
expect 206 "$R/threadpool/ThreadPool.cpp" 'double number = realGenerators\[tid\]\(\)'
sed -i '206a\	scs_ref_log_engine(0, number);' "$R/threadpool/ThreadPool.cpp"
expect 212 "$R/threadpool/ThreadPool.cpp" 'double number = intGenerators\[tid\]\(\)'
sed -i '212a\	scs_ref_log_engine(1, number);' "$R/threadpool/ThreadPool.cpp"
# MyDefine.cpp lines are +2 after patch 1 (two inserted returns above them)
expect 288 "$R/mydefine/MyDefine.cpp" 'rand\(\)/\(RAND_MAX'
sed -i '288s/rand()/scs_ref_rand()/' "$R/mydefine/MyDefine.cpp"
expect 293 "$R/mydefine/MyDefine.cpp" 'rand\(\)/\(RAND_MAX'
sed -i '293s/rand()/scs_ref_rand()/' "$R/mydefine/MyDefine.cpp"
expect 1512 "$R/profile/Profile.cpp" 'return v;'
sed -i '1512i\	scs_ref_log_gc(gc, v);' "$R/profile/Profile.cpp"
expect 1406 "$R/profile/Profile.cpp" 'unsigned seed = chrono'
sed -i '1406a\		seed = scs_ref_seed(2000 + l, seed);' "$R/profile/Profile.cpp"

build() {  # $1 = src dir, $2 = output binary, $3.. = extra flags / sources
    local src="$1" out="$2"; shift 2
    local inc=""; for d in $MODS; do inc="$inc -I$src/$d"; done
    local files="$src/scssim.cpp"
    for d in amplicon config fastahack fragment genome malbac mydefine profile seqwriter snp split threadpool vcfparser; do
        for f in "$src/$d"/*.cpp; do files="$files $f"; done
    done
    # FastaHack.cpp is the vendored tool's own main(); not part of scssim
    files="$(echo $files | tr ' ' '\n' | grep -v 'FastaHack.cpp' | tr '\n' ' ')"
    g++ -std=c++11 -O3 -DNDEBUG -w -pthread $inc "$@" $files -o "$out"
}
build "$S" "$OUT/bin/scssim" &
build "$R" "$OUT/bin/scssim_replay" -include "$HERE/ref_hooks.h" "$HERE/ref_hooks.cpp" &
wait
test -x "$OUT/bin/scssim" && test -x "$OUT/bin/scssim_replay"
echo "build_ref: built $OUT/bin/scssim and $OUT/bin/scssim_replay" >&2
