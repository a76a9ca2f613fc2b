#!/usr/bin/env bash
# TEST INFRASTRUCTURE — builds the *reference's own* hot-path code (read in place from
# /root/reference, never copied into this repo) plus oracle/ref_harness.cpp into
# oracle/_ref/libtrinity_ref.so.  Outputs ONLY under oracle/_ref/ (git-ignored, travels via gpurun).
#
# Two compile fixes are applied on the fly (g++ 13 instead of the reference's clang++):
#   1. queryexec_ctx.h:269-277 anonymous struct with std::vector members (clang extension):
#      a patched copy is *generated* into oracle/_ref/gen/ by the python snippet below.
#   2. boost spreadsort shim (oracle/shim/), snappy-stubs-public.h generated from its .in template.
# No reference build system (Makefile/cmake) is run.
set -euo pipefail
HERE="$(cd "$(dirname "$0")" && pwd)"
REF="${TRINITY_REFERENCE:-/root/reference}"
OUT="$HERE/_ref"
if [ ! -r "$REF/exec.cpp" ]; then
  if [ -f "$OUT/libtrinity_ref.so" ]; then echo "reference absent; using prebuilt $OUT/libtrinity_ref.so"; exit 0; fi
  # the tests compare with the reference's recorded outputs (tests/golden/reference_calls.json.gz) and skip what runs its code
  echo "reference sources not readable at $REF: oracle/_ref not built"; exit 0
fi
GEN="$OUT/gen"; OBJ="$OUT/obj"
rm -rf "$GEN" "$OBJ"; mkdir -p "$GEN" "$OBJ"
# symlink farm so that quote-includes resolve to the patched header first
for f in "$REF"/*.cpp "$REF"/*.h; do ln -s "$f" "$GEN/$(basename "$f")"; done
rm -f "$GEN/queryexec_ctx.h"
python3 - "$REF" "$GEN" <<'PY'
import re, sys
ref, gen = sys.argv[1], sys.argv[2]
src = open(f"{ref}/queryexec_ctx.h").read()
pat = re.compile(r"struct\s*\{\s*(#ifndef USE_BANKS.*?#endif\s*isrc_docid_t maxTrackedDocumentID\{0\}, lastMatchedDocumentID\{0\};)\s*\};", re.S)
new, n = pat.subn(lambda m: m.group(1), src)
assert n == 1, "anonymous-struct patch did not apply exactly once"
open(f"{gen}/queryexec_ctx.h", "w").write(new)
stub = open(f"{ref}/Switch/ext_snappy/snappy-stubs-public.h.in").read()
for k, v in {"${HAVE_SYS_UIO_H_01}": "1", "${PROJECT_VERSION_MAJOR}": "1", "${PROJECT_VERSION_MINOR}": "1", "${PROJECT_VERSION_PATCH}": "7"}.items():
    stub = stub.replace(k, v)
open(f"{gen}/snappy-stubs-public.h", "w").write(stub)
PY
ARCH="${TRINITY_REF_MARCH:-x86-64-v3}"
CXXF="-std=c++17 -fPIC -fno-rtti -Ofast -ffast-math -funroll-loops -march=$ARCH -fno-strict-aliasing -DLEAN_SWITCH -D_REENTRANT -w \
  -I$GEN -I$HERE/shim -I$REF -I$REF/Switch -I$REF/Switch/ext_snappy -I$REF/Switch/ext/FastPFor/headers"
TUS="google_codec lucene_codec docset_iterators docset_iterators_scorers docset_spans exec queryexec_ctx similarity codecs utils compilation_ctx queries index_source docwordspace docidupdates terms indexer segment_index_source merge"
pids=()
for t in $TUS; do
  g++ $CXXF -c "$GEN/$t.cpp" -o "$OBJ/$t.o" & pids+=($!)
done
g++ $CXXF -c "$REF/Switch/text.cpp" -o "$OBJ/switch_text.o" & pids+=($!)
for f in bitpacking bitpackingaligned bitpackingunaligned horizontalbitpacking simdbitpacking simdunalignedbitpacking; do
  g++ -O2 -fPIC -msse4.1 -w -I"$REF/Switch/ext/FastPFor/headers" -c "$REF/Switch/ext/FastPFor/src/$f.cpp" -o "$OBJ/fpf_$f.o" & pids+=($!)
done
# harness needs RTTI-free too (it subclasses reference types compiled -fno-rtti)
g++ $CXXF -c "$HERE/ref_harness.cpp" -o "$OBJ/ref_harness.o" & pids+=($!)
for p in "${pids[@]}"; do wait "$p"; done
g++ -shared -o "$OUT/libtrinity_ref.so" "$OBJ"/*.o -lpthread -lz
echo "built $OUT/libtrinity_ref.so"

# ---- second library: the SAME reference objects, except that exec_query() builds its span through the reference-side binding of
# libtrinity_b200.so (integration/gpu_exec.{h,cpp}, INTEGRATION.md) when the IndexSource has a device-resident twin.  The one call site
# (exec.cpp:1083-1086: build_iterator + build_span) is patched in a GENERATED copy of exec.cpp; nothing else of the reference changes.
B200LIB="$HERE/../trinity_b200/libtrinity_b200.so"
if [ -f "$B200LIB" ]; then
  python3 - "$REF" "$GEN" <<'PY'
import re, sys
ref, gen = sys.argv[1], sys.argv[2]
src = open(f"{ref}/exec.cpp").read()
pat = re.compile(r"auto \*const sit = rctx\.build_iterator\(rootExecNode, execFlags\);(.*?)auto\s+span\s+= build_span\(sit, &rctx\);", re.S)
def repl(m):
    return ("std::unique_ptr<DocsSetSpan> span = Trinity::b200_gpu_span(rctx, rootExecNode, execFlags, idxsrc, scorer);\n"
            "                        DocsSetIterators::Iterator *sit{nullptr};\n"
            "                        if (!span)\n"
            "                                sit = rctx.build_iterator(rootExecNode, execFlags);" + m.group(1) +
            "if (!span)\n                                span = build_span(sit, &rctx);")
new, n = pat.subn(repl, src)
assert n == 1, "exec_query span-site patch did not apply exactly once"
new = new.replace('#include "exec.h"', '#include "exec.h"\n#include "gpu_exec.h"', 1)
assert "gpu_exec.h" in new
open(f"{gen}/exec_gpu.cpp", "w").write(new)
PY
  INTEG="$HERE/../integration"
  gp=()
  g++ $CXXF -I"$INTEG" -c "$GEN/exec_gpu.cpp" -o "$OBJ/exec_gpu.o" & gp+=($!)
  g++ $CXXF -I"$INTEG" -c "$INTEG/gpu_exec.cpp" -o "$OBJ/gpu_exec.o" & gp+=($!)
  g++ $CXXF -I"$INTEG" -DTRINITY_B200_GPU_SPAN -c "$HERE/ref_harness.cpp" -o "$OBJ/ref_harness_gpu.o" & gp+=($!)
  for p in "${gp[@]}"; do wait "$p"; done
  objs=""
  for o in "$OBJ"/*.o; do
    case "$(basename "$o")" in exec.o|ref_harness.o) ;; *) objs="$objs $o";; esac
  done
  g++ -shared -o "$OUT/libtrinity_ref_gpu.so" $objs -L"$HERE/../trinity_b200" -ltrinity_b200 -Wl,-rpath,'$ORIGIN/../../trinity_b200' -lpthread -lz
  echo "built $OUT/libtrinity_ref_gpu.so"
fi
rm -rf "$GEN" "$OBJ"   # keep only the binaries under oracle/_ref/
