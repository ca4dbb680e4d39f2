#!/bin/bash
# Writes the SASS of the hot kernels (c3 = bf16, prob bits 10) to profiles/rNN_sass_<kernel>.txt and a summary
# of the Blackwell-specific mnemonics per kernel (UBLKCP = cp.async.bulk / TMA 1-D, LDGSTS = cp.async,
# SYNCS = mbarrier, ATOMS.POPC.INC = warp-aggregated shared atomic).  usage: tools/sass_dump.sh r02
set -e
tag=${1:-r02}
cd "$(dirname "$0")/.."
O=dietgpu_b200/csrc/build
dump() {  # object, function-name regex, output name
  cuobjdump -sass $O/$1.o | awk -v pat="$2" '/Function : /{f = ($0 ~ pat)} f' | grep -v '^\s*/\* 0x' | sed -E 's#\s*/\* 0x[0-9a-f]+ \*/##' > profiles/${tag}_sass_$3.txt
  echo "$3: $(wc -l < profiles/${tag}_sass_$3.txt) lines"
}
dump encode 'statsFloatKernelILi2EE' stats_bf16
dump encode 'statsBytesKernelE' stats_bytes
dump encode 'encodeKernelFastILb0ELi0' encode_bytes_packed
dump encode 'encodeKernelFastILb1ELi2' encode_bf16_wide
dump decode 'decodeFusedKernelILi2ELi10ELi8' decode_bf16_pb10
dump decode 'decodeFusedKernelILi0ELi10ELi8' decode_bytes_pb10
{
  echo "# Blackwell / async mnemonics per hot kernel (counts of SASS instructions), libdietgpu_b200.so build of $(git rev-parse --short HEAD)"
  for f in profiles/${tag}_sass_*.txt; do
    case $f in *_sass_summary.txt) continue;; esac
    printf "%s:" "$(basename $f .txt)"
    for m in UBLKCP UTMALDG LDGSTS SYNCS ATOMS.POPC.INC VOTE.ANY VOTEU POPC UPOPC 'LDS.128' 'LDS.64' 'STG.E.128' 'STG.E.64' 'LDG.E.128' LEA.HI IMAD.HI; do
      printf " %s=%s" "$m" "$(grep -c -- "$m" $f || true)"
    done
    echo
  done
} > profiles/${tag}_sass_summary.txt
cat profiles/${tag}_sass_summary.txt
