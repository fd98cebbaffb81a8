#!/bin/bash
# SASS evidence of the Blackwell-native paths: counts of the tcgen05 / TMA mnemonics per object
# (B200_PROFILING.md: tcgen05.mma -> UTCHMMA, tcgen05.ld/st -> LDTM/STTM, cp.async.bulk -> UBLKCP).
#   bash profiles/scripts/sass_counts.sh > profiles/r02_sass.md     (after `make -C dynibar_b200/csrc`)
cd "$(dirname "$0")/../../dynibar_b200/csrc"
echo "# r02 — SASS mnemonic counts per object (\`cuobjdump -sass <obj> | grep -c <mnemonic>\`)"
echo
echo "Built with \`nvcc -gencode arch=compute_100a,code=sm_100a\` (csrc/Makefile). \`UTCHMMA\` = \`tcgen05.mma.kind::f16\`,"
echo "\`LDTM\` / \`STTM\` = \`tcgen05.ld\` / \`tcgen05.st\`, \`UBLKCP\` = \`cp.async.bulk\` (TMA engine, non-tensor form),"
echo "\`SYNCS\` = mbarrier operations, \`MUFU.EX2\` = the ELU / softmax exponentials. No \`HMMA\` (legacy mma.sync) other than"
echo "as a substring of \`UTCHMMA\`; no \`UTMALDG\` (the bulk copies are 1-D: weight chunks and activation tile images)."
echo
echo "| object | UTCHMMA | LDTM | STTM | UBLKCP | UTMALDG | SYNCS | MUFU.EX2 | legacy HMMA |"
echo "|---|---|---|---|---|---|---|---|---|"
for f in view_twin3 chains_twin chains_fused attention_tc linear_tc train_tc; do
  cuobjdump -sass $f.o > /tmp/_sass_$f.txt 2>/dev/null
  c() { grep -c "$1" /tmp/_sass_$f.txt; }
  legacy=$(grep "HMMA" /tmp/_sass_$f.txt | grep -vc "UTCHMMA")
  echo "| \`$f.o\` | $(c UTCHMMA) | $(c LDTM) | $(c STTM) | $(c UBLKCP) | $(c UTMALDG) | $(c SYNCS) | $(c 'MUFU.EX2') | $legacy |"
done
