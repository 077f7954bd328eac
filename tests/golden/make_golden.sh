#!/bin/sh
# Regenerates the golden GAF files from the UNMODIFIED reference (oracle/_ref/minigraph, built by oracle/Makefile from
# /root/reference). Inputs are produced by tools/mgsim (deterministic, splitmix64) so only the expected outputs are stored.
set -e
cd "$(dirname "$0")/../.."
R=oracle/_ref/minigraph; S=tools/mgsim; G=tests/golden; F=$G/fixtures; T=$(mktemp -d)
$R -cx lr $F/MT.gfa $F/MT-orangA.fa 2>/dev/null > $G/c1_MT_orangA.lr.gaf
$R -cx lr $F/MT.gfa $F/MT-chimp.fa 2>/dev/null > $G/c1_MT_chimp.lr.gaf
$S walk -g $F/MT.gfa -w ">MTh0>MTh4001>MTh4502>MTh9505>MTh13014>MTh13516" -w ">MTh0<MTo3426>MTh4502>MTo8961>MTh9505>MTh13516" -o $T/mt.hap.fa
$S reads -i $T/mt.hap.fa -n 24 -l 10000 -e ont -s 11 -o $T/mt.reads.fa 2>/dev/null
$R -cx lr $F/MT.gfa $T/mt.reads.fa 2>/dev/null > $G/c2_MT_24x10k_ont_s11.lr.gaf
$S graph -l 300000 -n 3 -s 7 -o $T/sv 2>/dev/null
$S reads -i $T/sv.hap.fa -n 24 -l 15000 -e ont -s 5 -o $T/sv.reads.fa 2>/dev/null
$R -cx lr $T/sv.gfa $T/sv.reads.fa 2>/dev/null > $G/c3_sv300k_h3_s7_24x15k_ont_s5.lr.gaf
$S reads -i $F/MT-human.fa -n 12 -l 20000 -e hifi -s 13 -c -o $T/mth.reads.fa 2>/dev/null
$R -cx asm $F/MT-human.fa $T/mth.reads.fa 2>/dev/null > $G/c4_MThuman_12x20k_hifi_s13.asm.gaf
rm -rf $T
md5sum $G/*.gaf
# larger sets (gzip -n: byte-stable archives): 240 / 240 / 200 reads, the SV graph at the density of the MHC-scale bench graph
T=$(mktemp -d)
$S walk -g $F/MT.gfa -w ">MTh0>MTh4001>MTh4502>MTh9505>MTh13014>MTh13516" -w ">MTh0<MTo3426>MTh4502>MTo8961>MTh9505>MTh13516" -o $T/mt.hap.fa
$S reads -i $T/mt.hap.fa -n 240 -l 10000 -e ont -s 111 -o $T/mt.reads.fa 2>/dev/null
$R -cx lr -t 8 $F/MT.gfa $T/mt.reads.fa 2>/dev/null | gzip -n9 > $G/L2_MT_240x10k_ont_s111.lr.gaf.gz
$S graph -l 1000000 -n 8 -s 7 -o $T/sv 2>/dev/null
$S reads -i $T/sv.hap.fa -n 240 -l 15000 -e ont -s 105 -o $T/sv.reads.fa 2>/dev/null
# 3 MB of GAF text: kept as one 64-bit BLAKE2b digest per line
$R -cx lr -t 8 $T/sv.gfa $T/sv.reads.fa 2>/dev/null | python3 -c 'import hashlib, sys
for ln in sys.stdin.buffer: print(hashlib.blake2b(ln.rstrip(b"\n"), digest_size=8).hexdigest())' > $G/L3_sv1m_h8_s7_240x15k_ont_s105.lr.gaf.b2
$S reads -i $F/MT-human.fa -n 200 -l 20000 -e hifi -s 113 -c -o $T/mth.reads.fa 2>/dev/null
$R -cx asm -t 8 $F/MT-human.fa $T/mth.reads.fa 2>/dev/null | gzip -n9 > $G/L4_MThuman_200x20k_hifi_s113.asm.gaf.gz
rm -rf $T
ls -la $G/*.gz $G/*.b2
