#!/bin/bash
# Builds the host-emulated library + the pybind module against it into tools/emu/build/ (development tooling).
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
ROOT="$(cd "$HERE/../.." && pwd)"
CSRC="$ROOT/quantized_decoder_polar_codes_b200/csrc"
OUT="$HERE/build"
mkdir -p "$OUT"
OPT="${PB_EMU_OPT:--O1}"
g++ $OPT -g -std=c++17 -fPIC -shared -w -ffp-contract=off -x c++ -I"$HERE/shim" -I"$CSRC" "$HERE/emu_lib.cpp" -o "$OUT/libpolar_b200.so"
PYINC=$(python -c "import importlib.util as u,sysconfig;s=u.spec_from_file_location('pb_build','$ROOT/quantized_decoder_polar_codes_b200/build.py');m=u.module_from_spec(s);s.loader.exec_module(m);print('-I'+sysconfig.get_paths()['include']+' -I'+m.pybind11_include())")
EXT=$(python -c "import sysconfig;print(sysconfig.get_config_var('EXT_SUFFIX'))")
if [ ! -f "$OUT/_libPolarDecoder$EXT" ] || [ "$CSRC/pb_pybind.cpp" -nt "$OUT/_libPolarDecoder$EXT" ]; then
  g++ -O1 -std=c++17 -fPIC -shared -fvisibility=hidden $PYINC "$CSRC/pb_pybind.cpp" -L"$OUT" -lpolar_b200 -Wl,-rpath,'$ORIGIN' -o "$OUT/_libPolarDecoder$EXT"
fi
echo "built $OUT"
