#!/usr/bin/env bash
# Regenerates the golden fixtures in this directory by running the UNMODIFIED reference binary
# (oracle/_ref/plink2 / plink2_lapack, built by oracle/build_ref.sh from /root/reference).
# The reference ships no golden vectors for KING / GRM / --indep-pairwise (SURVEY.md section 4), so
# these outputs of the reference itself are what pins the oracle (oracle/plink_oracle.py) and,
# through it, the CUDA path.  Run from the repo root: bash tests/golden/make_golden.sh
set -euo pipefail
cd "$(dirname "$0")"
P=../../oracle/_ref/plink2
PL=../../oracle/_ref/plink2_lapack
T=$(mktemp -d)
# --- set A: 100 samples x 1000 variants, 3% missing, HWE genotypes, ~half the variants in LD with
# their predecessor (2.0/plink2_import.cc:16326-16460).  --dummy output depends on --threads.
$P --dummy 100 1000 0.03 --seed 7 --threads 2 --make-bed --out $T/a > /dev/null
cp $T/a.bed a.bed; cp $T/a.bim a.bim; cp $T/a.fam a.fam
$P --bfile a --make-pgen --out $T/a_pgen --threads 2 > /dev/null        # mode 0x10 (difflist / LD-compressed records)
cp $T/a_pgen.pgen a_mode10.pgen
$P --bfile a --make-pgen format=2 --out $T/a_f2 --threads 2 > /dev/null  # mode 0x02 fixed width
cp $T/a_f2.pgen a_mode02.pgen; cp $T/a_f2.pvar a.pvar; cp $T/a_f2.psam a.psam
$P --bfile a --make-king-table counts cols=+ibs1,+ibs --make-king bin4 triangle --threads 2 --out $T/a_king > /dev/null
gzip -9 -n -c $T/a_king.kin0 > a_king.kin0.gz; cp $T/a_king.king.bin a_king.king.bin
$P --bfile a --make-king-table --threads 2 --out $T/a_kingp > /dev/null   # default proportion columns
gzip -9 -n -c $T/a_kingp.kin0 > a_kingp.kin0.gz
$P --bfile a --make-king square --threads 2 --out $T/a_kingsq > /dev/null
gzip -9 -n -c $T/a_kingsq.king > a_kingsq.king.gz; cp $T/a_kingsq.king.id a_kingsq.king.id
$P --bfile a --make-king-table counts --parallel 2 3 --threads 2 --out $T/a_kingpar > /dev/null
gzip -9 -n -c $T/a_kingpar.kin0.2 > a_kingpar.kin0.2.gz
$P --bfile a --make-king-table counts --king-table-filter 0.02 --threads 2 --out $T/a_kf > /dev/null
cp $T/a_kf.kin0 a_kingfilt.kin0
# pair-list KING (--king-table-subset): (1) the proportion table above as the pair list with a kinship threshold,
# (2) a hand-written IID-only list with swapped orientation, an unknown ID and ibs1 columns
zcat a_kingp.kin0.gz > $T/in.kin0
$P --bfile a --make-king-table counts --king-table-subset $T/in.kin0 -0.05 --threads 2 --out $T/a_sub > /dev/null
gzip -9 -n -c $T/a_sub.kin0 > a_kingsub.kin0.gz
printf '#IID1\tIID2\tKINSHIP\nper7\tper3\t0.1\nper2\tper90\t0.2\nnosuch\tper1\t0.3\nper50\tper49\t-0.4\n' > a_sub2.txt
$P --bfile a --make-king-table counts cols=+ibs1 --king-table-subset a_sub2.txt --threads 2 --out $T/a_sub2 > /dev/null
cp $T/a_sub2.kin0 a_kingsub2.kin0
$P --bfile a --king-cutoff 0.02 --threads 2 --out $T/a_cut > /dev/null
cp $T/a_cut.king.cutoff.in.id a_cut.king.cutoff.in.id; cp $T/a_cut.king.cutoff.out.id a_cut.king.cutoff.out.id
$P --bfile a --freq --threads 2 --out $T/a_freq > /dev/null
cp $T/a_freq.afreq a.afreq
$P --pgen a_mode02.pgen --pvar a.pvar --psam a.psam --freq --threads 2 --out $T/a_pf > /dev/null   # REF not provisional: no PROVISIONAL_REF? column
cp $T/a_pf.afreq a_pvar.afreq
$P --bfile a --make-grm-bin --threads 2 --out $T/a_grm > /dev/null
cp $T/a_grm.grm.bin a_grm.grm.bin; cp $T/a_grm.grm.N.bin a_grm.grm.N.bin; cp $T/a_grm.grm.id a_grm.grm.id
$P --bfile a --make-grm-bin meanimpute --threads 2 --out $T/a_grmmi > /dev/null
$P --bfile a --make-grm-list --threads 2 --out $T/a_grml > /dev/null
gzip -9 -n -c $T/a_grml.grm > a_grml.grm.gz
$P --bfile a --make-grm-sparse 0.02 --threads 2 --out $T/a_sp > /dev/null
cp $T/a_sp.grm.sp a_grmsp.grm.sp
cp $T/a_grmmi.grm.bin a_grmmi.grm.bin
$P --bfile a --make-rel cov bin4 triangle --threads 2 --out $T/a_relcov > /dev/null
cp $T/a_relcov.rel.bin a_relcov.rel.bin
$P --bfile a --make-rel square --threads 2 --out $T/a_rel > /dev/null
gzip -9 -n -c $T/a_rel.rel > a_rel.rel.gz
$P --bfile a --indep-pairwise 50 5 0.2 --threads 2 --out $T/a_ld > /dev/null
cp $T/a_ld.prune.in a_ld.prune.in; cp $T/a_ld.prune.out a_ld.prune.out
$P --bfile a --indep-pairwise 100 1 0.1 --threads 2 --out $T/a_ld2 > /dev/null
cp $T/a_ld2.prune.in a_ld2.prune.in
$P --bfile a --indep-pairwise 20kb 0.3 --threads 2 --out $T/a_ldkb > /dev/null
awk 'NR%7==3{print $2}' a.bim > a_pref.txt
$P --bfile a --indep-pairwise 50 5 0.1 --indep-preferred a_pref.txt --threads 2 --out $T/a_ldp > /dev/null
cp $T/a_ldp.prune.in a_ldpref.prune.in
cp $T/a_ldkb.prune.in a_ldkb.prune.in
$P --bfile a --indep-pairwise 50 5 0.2 --indep-order 1 --threads 2 --out $T/a_ldo1 > /dev/null
cp $T/a_ldo1.prune.in a_ldo1.prune.in
# --score: shuffled (variant, allele, weight) lines incl. unknown IDs / foreign allele codes (make_score_set.py)
python make_score_set.py a.bim a_score.txt
$P --bfile a --score a_score.txt header --threads 2 --out $T/a_sc > /dev/null
$P --bfile a --score a_score.txt header no-mean-imputation cols=+scoresums,+denom --threads 2 --out $T/a_sc2 > /dev/null
cp $T/a_sc.sscore a_sc.sscore; cp $T/a_sc2.sscore a_sc2.sscore
$P --bfile a --score a_score.txt header center cols=+scoresums --threads 2 --out $T/a_scc > /dev/null
$P --bfile a --score a_score.txt header variance-standardize cols=+scoresums --threads 2 --out $T/a_scv > /dev/null
cp $T/a_scc.sscore a_sc_center.sscore; cp $T/a_scv.sscore a_sc_varstd.sscore
$P --bfile a --score a_score.txt header dominant list-variants cols=+scoresums,+denom --threads 2 --out $T/a_scd > /dev/null
$P --bfile a --score a_score.txt header recessive cols=+scoresums,+denom --threads 2 --out $T/a_scr > /dev/null
cp $T/a_scd.sscore a_sc_dominant.sscore; cp $T/a_scr.sscore a_sc_recessive.sscore; cp $T/a_scd.sscore.vars a_sc.sscore.vars
# --variant-score: two weight columns for 89 of the 100 samples + one unknown ID (a_vscore_weights.txt is kept as written)
$P --bfile a --variant-score a_vscore_weights.txt --threads 2 --out $T/a_vs > /dev/null
$P --bfile a --variant-score a_vscore_weights.txt cols=+altfreq --threads 2 --out $T/a_vsf > /dev/null
cp $T/a_vs.vscore a_vs.vscore; cp $T/a_vsf.vscore a_vs_altfreq.vscore
# --king-cutoff-table on the proportion table written above
$P --bfile a --king-cutoff-table $T/in.kin0 0.02 --threads 2 --out $T/a_kct > /dev/null
cp $T/a_kct.king.cutoff.in.id a_kct.king.cutoff.in.id; cp $T/a_kct.king.cutoff.out.id a_kct.king.cutoff.out.id
# --king-cutoff <prefix> <threshold>: (1) the fp32 triangle written above (a_king.king.bin + a_kingsq.king.id),
# (2) an fp64 triangle over a shuffled 80-ID subset with unknown IDs mixed in (make_king_cutoff_set.py)
cp a_king.king.bin $T/kc4.king.bin; cp a_kingsq.king.id $T/kc4.king.id
$P --bfile a --king-cutoff $T/kc4 0.02 --threads 2 --out $T/a_kc4 > /dev/null
cp $T/a_kc4.king.cutoff.in.id a_kc4.king.cutoff.in.id; cp $T/a_kc4.king.cutoff.out.id a_kc4.king.cutoff.out.id
$P --bfile a --make-king bin triangle --threads 2 --out $T/k8 > /dev/null
python make_king_cutoff_set.py $T/k8.king.bin $T/k8.king.id a_kc8
$P --bfile a --king-cutoff a_kc8 0.03 --threads 2 --out $T/a_kc8o > /dev/null
cp $T/a_kc8o.king.cutoff.in.id a_kc8.king.cutoff.in.id; cp $T/a_kc8o.king.cutoff.out.id a_kc8.king.cutoff.out.id
# --- filters in front of the commands, pinned through --make-bed (host-only): ID lists from make_filter_set.py
python make_filter_set.py
$P --bfile x --keep x_keep1.txt x_keep2.txt --remove x_remove.txt --extract x_extract.txt --exclude x_exclude.txt --make-bed --threads 2 --out $T/x_filt > /dev/null
for e in bed bim fam; do cp $T/x_filt.$e x_filt.$e; done
$P --bfile x --keep x_keep1.txt x_keep2.txt --remove x_remove.txt --extract x_extract.txt --exclude x_exclude.txt --keep-founders --make-bed --threads 2 --out $T/x_ff > /dev/null
cp $T/x_ff.bed x_filt_founders.bed   # founders of the filtered view: what the founder-only commands decode
$P --bfile x --chr 1,X,Y --not-chr Y --make-bed --threads 2 --out $T/x_chr > /dev/null
cp $T/x_chr.bim x_chr.bim; cp $T/x_chr.bed x_chr.bed
$P --pgen a_mode10.pgen --pvar a.pvar --psam a.psam --remove x_remove.txt --exclude x_exclude.txt --make-bed --threads 2 --out $T/a_filt > /dev/null
for e in bed bim fam; do cp $T/a_filt.$e a_filt.$e; done
$P --bfile s --keep-fam s_keepfam.txt --remove-fam s_removefam.txt --make-bed --threads 2 --out $T/s_fam > /dev/null
cp $T/s_fam.fam s_famfilt.fam; cp $T/s_fam.bed s_famfilt.bed
# count-based QC thresholds (--mind, --geno, --maf / --max-maf / --mac) and the sex / founder filters
$P --bfile x --keep x_keep1.txt x_keep2.txt --mind 0.035 --geno 0.02 --maf 0.05 --make-bed --threads 2 --out $T/x_qc > /dev/null
for e in bed bim fam mindrem.id; do cp $T/x_qc.$e x_qc.$e; done
$P --bfile x --keep-founders --mac 30 --max-maf 0.45 --make-bed --threads 2 --out $T/x_mac > /dev/null; cp $T/x_mac.bim x_mac.bim; cp $T/x_mac.fam x_mac.fam
$P --bfile x --remove-nosex --keep-nonfounders --make-bed --threads 2 --out $T/x_sex > /dev/null; cp $T/x_sex.fam x_sex.fam
$P --pgen a_mode10.pgen --pvar a.pvar --psam a.psam --geno 0.03 --mind 0.04 --maf 0.2 --make-bed --threads 2 --out $T/a_qc > /dev/null
for e in bed bim fam; do cp $T/a_qc.$e a_qc.$e; done
$P --bfile a --read-freq a_rf.afreq --exclude x_exclude.txt --maf 0.3 --make-bed --threads 2 --out $T/a_rfmaf > /dev/null; cp $T/a_rfmaf.bim a_rfmaf.bim   # --maf on loaded frequencies
# --snps-only [just-acgt] on awkward allele codes (x_alleles.bim), --from-kb/--to-kb, --write-snplist / --write-samples
$P --bed x.bed --bim x_alleles.bim --fam x.fam --snps-only --make-bed --threads 2 --out $T/s1 > /dev/null; cp $T/s1.bim x_snps.bim
$P --bed x.bed --bim x_alleles.bim --fam x.fam --snps-only just-acgt --make-bed --threads 2 --out $T/s2 > /dev/null; cp $T/s2.bim x_acgt.bim
$P --bfile x --chr 1 --from-kb 0.1001 --to-kb 0.25 --keep x_keep2.txt --write-snplist --write-samples --threads 2 --out $T/s3 > /dev/null; cp $T/s3.snplist x_bp.snplist; cp $T/s3.id x_bp.id
$P --bfile x --make-pgen vzs --threads 2 --out $T/xz > /dev/null; cp $T/xz.pvar.zst x.pvar.zst   # Zstandard-compressed .pvar as the reference writes it
# --nonfounders: allele frequencies (thresholds, --freq report, LD tie-breaks) from all 120 samples of set X, not its 116 founders
$P --bfile x --nonfounders --maf 0.1 --mac 30 --make-bed --threads 2 --out $T/n1 > /dev/null; cp $T/n1.bim x_nf.bim
$P --bfile x --nonfounders --freq --threads 2 --out $T/n2 > /dev/null; cp $T/n2.afreq x_nf.afreq
$P --bfile x --nonfounders --freq counts --threads 2 --out $T/n4 > /dev/null; cp $T/n4.acount x_nf.acount
$P --bfile x --chr 1 --nonfounders --indep-pairwise 50 5 0.2 --threads 2 --out $T/n3 > /dev/null; cp $T/n3.prune.in x_nf.prune.in
# --set-missing-var-ids on a .bim whose every third ID is '.' (alleles incl. '0' codes, multi-character and symbolic ones)
awk 'BEGIN{OFS="\t"} {if (NR%3==0) $2="."; print}' x_alleles.bim > x_noid.bim
$P --bed x.bed --bim x_noid.bim --fam x.fam --set-missing-var-ids '@:#:$1:$2' --make-bed --threads 2 --out $T/v1 > /dev/null; cp $T/v1.bim x_setid.bim
# --allow-extra-chr: set X with its XY block renamed chrUn_KI270 and half of MT renamed GL000.1 (diploid, autosome-like contigs)
awk 'BEGIN{OFS="\t"} {if ($1=="XY") $1="chrUn_KI270"; if ($1=="MT" && ++k<=50) $1="GL000.1"; print}' x.bim > x_contigs.bim
$P --bed x.bed --bim x_contigs.bim --fam x.fam --allow-extra-chr --not-chr 1,X --make-bed --threads 2 --out $T/e1 > /dev/null; cp $T/e1.bim x_contigs_sub.bim
$P --bed x.bed --bim x_contigs.bim --fam x.fam --allow-extra-chr --not-chr X,Y,MT --indep-pairwise 50 5 0.2 --threads 2 --out $T/e2 > /dev/null; cp $T/e2.prune.in x_contigs.prune.in
$P --bed x.bed --bim x_contigs.bim --fam x.fam --allow-extra-chr --make-king-table --threads 2 --out $T/e3 > /dev/null; gzip -9 -n -c $T/e3.kin0 > x_contigs.kin0.gz
# --make-pgen: the reference's .pvar / .psam text, its fixed-width .pgen (format=2; the default mode is compressed
# differently and not compared) + the .bed of the same view
$P --bfile x --keep x_keep1.txt x_keep2.txt --extract x_extract.txt --make-pgen --threads 2 --out $T/mp > /dev/null; cp $T/mp.pvar x_mp.pvar; cp $T/mp.psam x_mp.psam
$P --bfile x --keep x_keep1.txt x_keep2.txt --extract x_extract.txt --make-bed --threads 2 --out $T/mb > /dev/null; cp $T/mb.bed x_mp.bed
$P --bfile x --keep x_keep1.txt x_keep2.txt --extract x_extract.txt --make-pgen format=2 --threads 2 --out $T/mpf2 > /dev/null; cp $T/mpf2.pgen x_mp.pgen
$P --pedmap p --make-pgen --threads 2 --out $T/pp > /dev/null; cp $T/pp.pvar p_mp.pvar; cp $T/pp.psam p_mp.psam
$P --bfile x --bp-space 7 --maf 0.05 --chr 1,X,MT --make-bed --threads 2 --out $T/bs > /dev/null; cp $T/bs.bim x_bpspace.bim   # --bp-space runs after the frequency thresholds
# --missing: written after the sample filters (incl. --mind) and before the variant thresholds
$P --bfile x --keep x_keep1.txt x_keep2.txt --mind 0.05 --geno 0.05 --missing --threads 2 --out $T/ms > /dev/null; cp $T/ms.smiss x_miss.smiss; cp $T/ms.vmiss x_miss.vmiss
# relatedness prune from a table, then --make-bed on the survivors
$P --bfile a --king-cutoff-table $T/in.kin0 0.02 --make-bed --threads 2 --out $T/a_kctb > /dev/null
cp $T/a_kctb.fam a_kctb.fam; cp $T/a_kctb.bed a_kctb.bed
# the same filters / prune chaining through the device commands (tests/test_filters_gpu.py, tools/check_r2s.py)
XF="--keep x_keep1.txt x_keep2.txt --remove x_remove.txt --extract x_extract.txt --exclude x_exclude.txt"
$P --bfile x $XF --make-king-table --threads 2 --out $T/g1 > /dev/null; gzip -9 -n -c $T/g1.kin0 > g_xfilt.kin0.gz
$P --bfile x $XF --indep-pairwise 50 5 0.2 --threads 2 --out $T/g2 > /dev/null; cp $T/g2.prune.in g_xfilt.prune.in
$P --bfile x $XF --freq --threads 2 --out $T/g3 > /dev/null; cp $T/g3.afreq g_xfilt.afreq
$P --bfile a --king-cutoff 0.02 --indep-pairwise 50 5 0.2 --threads 2 --out $T/g4 > /dev/null; cp $T/g4.prune.in g_acut.prune.in
$P --bfile a --king-cutoff 0.02 --make-grm-bin --threads 2 --out $T/g5 > /dev/null; cp $T/g5.grm.bin g_acut.grm.bin
$PL --bfile a --king-cutoff-table $T/in.kin0 0.02 --pca 3 --threads 2 --out $T/g6 > /dev/null; cp $T/g6.eigenval g_akct.eigenval; cp $T/g6.eigenvec g_akct.eigenvec
$P --pgen a_mode10.pgen --pvar a.pvar --psam a.psam --remove x_remove.txt --exclude x_exclude.txt --make-king-table --threads 2 --out $T/g7 > /dev/null; gzip -9 -n -c $T/g7.kin0 > g_afilt.kin0.gz
$P --bfile a --king-cutoff 0.02 --score a_score.txt header cols=+scoresums,+denom --threads 2 --out $T/g8 > /dev/null; cp $T/g8.sscore g_acut.sscore
# host orchestration of the LD prune, replayed on the CPU through tests/harness/mock_pl2gpu.cc: several chromosome runs of
# uneven length (one of them a singleton), a prune chained behind --king-cutoff-table, a filtered view
awk 'BEGIN{OFS="\t"} {c=(NR<=120)?1:(NR<=480)?2:(NR<=500)?3:(NR<=501)?4:(NR<=800)?5:7; $1=c; print}' a.bim > a_chr6.bim
$P --bed a.bed --bim a_chr6.bim --fam a.fam --indep-pairwise 50 5 0.2 --threads 2 --out $T/c6 > /dev/null; cp $T/c6.prune.in a_chr6.prune.in
$P --bfile a --king-cutoff-table $T/in.kin0 0.02 --indep-pairwise 50 5 0.2 --threads 2 --out $T/kl > /dev/null; cp $T/kl.prune.in g_akct.prune.in
$P --bfile a --remove x_remove.txt --exclude x_exclude.txt --indep-pairwise 50 5 0.2 --threads 2 --out $T/fl > /dev/null; cp $T/fl.prune.in g_afilt.prune.in
# --r2-unphased tables: all pairs of set A at the default filters, a 7-variant / r^2 >= 0.5 window, and set X without chrX
# under --keep (chrY: female founders count as missing; MT / XY like autosomes; non-founders ignored)
$P --bfile a --r2-unphased --threads 2 --out $T/r1 > /dev/null; gzip -9 -n -c $T/r1.vcor > a_r2.vcor.gz
$P --bfile a --r2-unphased --ld-window 7 --ld-window-r2 0.5 --threads 2 --out $T/r2 > /dev/null; gzip -9 -n -c $T/r2.vcor > a_r2w.vcor.gz
$P --bfile x --not-chr X --keep x_keep1.txt x_keep2.txt --r2-unphased --ld-window-r2 0.3 --ld-window-kb 0.1 --threads 2 --out $T/r3 > /dev/null; gzip -9 -n -c $T/r3.vcor > x_r2.vcor.gz
# chrX r^2 (male-downweighted statistic, non-major-allele coding): set X under --keep with every chromosome, and --nonfounders on X + Y
$P --bfile x --keep x_keep1.txt x_keep2.txt --r2-unphased --ld-window-r2 0.1 --ld-window-kb 0.05 --threads 2 --out $T/r4 > /dev/null; gzip -9 -n -c $T/r4.vcor > x_r2x.vcor.gz
$P --bfile x --nonfounders --r2-unphased --ld-window-r2 0.1 --chr X,Y --threads 2 --out $T/r5 > /dev/null; gzip -9 -n -c $T/r5.vcor > x_r2nf.vcor.gz
# --read-freq: a perturbed / partial / allele-swapped copy of a.afreq (make_read_freq_set.py)
python make_read_freq_set.py a.afreq a_rf.afreq
$P --bfile a --read-freq a_rf.afreq --make-grm-bin --threads 2 --out $T/a_rf > /dev/null
$P --bfile a --read-freq a_rf.afreq --indep-pairwise 50 5 0.2 --threads 2 --out $T/a_rfld > /dev/null
cp $T/a_rf.grm.bin a_rf.grm.bin; cp $T/a_rfld.prune.in a_rfld.prune.in
# --- set X: chromosomes 1 / X / Y / XY / MT with mixed sexes and non-founders (make_x_set.py): the sex-chromosome
# forms of --indep-pairwise, both pruning orders
$P --dummy 120 800 0.03 --seed 11 --threads 2 --make-bed --out $T/x0 > /dev/null
python make_x_set.py $T/x0 x
$P --bfile x --indep-pairwise 50 5 0.2 --threads 2 --out $T/x_o2 > /dev/null
$P --bfile x --indep-pairwise 50 5 0.2 --indep-order 1 --threads 2 --out $T/x_o1 > /dev/null
cp $T/x_o2.prune.in x_o2.prune.in; cp $T/x_o1.prune.in x_o1.prune.in
$P --bfile x --indep-pairwise 30kb 0.3 --threads 2 --out $T/x_kb > /dev/null
cp $T/x_kb.prune.in x_kb.prune.in
$P --bfile x --freq --threads 2 --out $T/x_f > /dev/null
cp $T/x_f.afreq x.afreq
# rel-check: sets R (60 samples, 2 FIDs, IIDs chosen to exercise the natural sort: leading zeros, mixed case, digit runs)
# and S (300 random IDs over 5 FIDs) are kept as written by the script that made them (tests/golden/README in DESIGN 7)
$P --bfile r --make-king-table rel-check counts --threads 2 --out $T/r_rc > /dev/null
cp $T/r_rc.kin0 r_relcheck.kin0
$P --bfile s --make-king-table rel-check --threads 2 --out $T/s_rc > /dev/null
gzip -9 -n -c $T/s_rc.kin0 > s_relcheck.kin0.gz
if [ -x $PL ]; then
  $PL --bfile a --pca 4 --threads 2 --out $T/a_pca > /dev/null
  cp $T/a_pca.eigenval a_pca.eigenval; cp $T/a_pca.eigenvec a_pca.eigenvec
  $PL --bfile a --pca 3 approx --seed 11 --threads 2 --out $T/a_pcaa > /dev/null
  cp $T/a_pcaa.eigenval a_pcaa.eigenval; cp $T/a_pcaa.eigenvec a_pcaa.eigenvec
fi
# --- set P: legacy text filesets (make_ped_set.py) through the reference's --pedmap import
python make_ped_set.py
$P --pedmap p --make-bed --threads 2 --out $T/p > /dev/null; for e in bed bim fam; do cp $T/p.$e p.$e; done
$P --ped pc.ped --map pc.map --make-bed --threads 2 --out $T/pc > /dev/null; cp $T/pc.bed pc.bed; cp $T/pc.bim pc.bim
# --- set MA: a .pgen with multiallelic records, one of them the LD base of a biallelic record (make_multiallelic_set.py)
python make_multiallelic_set.py
$P --vcf ma.vcf --make-pgen --threads 2 --out $T/ma > /dev/null; cp $T/ma.pgen ma.pgen; cp $T/ma.pvar ma.pvar; cp $T/ma.psam ma.psam; rm ma.vcf
$P --pfile ma --max-alleles 2 --make-bed --threads 2 --out $T/ma_bi > /dev/null; cp $T/ma_bi.bed ma_bi.bed; cp $T/ma_bi.bim ma_bi.bim
# --- set T: the reference's own toy fixture (1.9/toy.ped + toy.map; BASELINE.json configs[0])
if [ -f /root/reference/1.9/toy.ped ]; then
  $P --ped /root/reference/1.9/toy.ped --map /root/reference/1.9/toy.map --make-bed --out $T/toy > /dev/null
  cp $T/toy.bed toy.bed; cp $T/toy.bim toy.bim; cp $T/toy.fam toy.fam
  $P --bfile toy --make-king square --make-king-table counts cols=+ibs1,+ibs --out $T/toy_king > /dev/null
  cp $T/toy_king.king toy_king.king; cp $T/toy_king.kin0 toy_king.kin0
fi
rm -rf $T
ls -la

# --- set B: structure-rich reader fixture (37 samples, 400 variants): rare-ALT / rare-REF variants (difflists on
# either base), monomorphic and all-missing variants, 40 % missingness, near-copies of the previous variant
# (LD-compressed records).  The .bed is synthesised here, the .pgen is written by the reference.
python3 - <<'PY'
import numpy as np
rng = np.random.default_rng(99)
n, m = 37, 400
g = np.zeros((m, n), dtype=np.uint8)
for v in range(m):
    kind = v % 8
    f = {0: 0.5, 1: 0.01, 2: 0.01, 3: 0.99, 4: 0.0}.get(kind, None)
    if f is None:
        f = rng.uniform(0.02, 0.98)
    g[v] = (rng.random(n) < f).astype(np.uint8) + (rng.random(n) < f)
    if kind == 5:
        g[v][rng.random(n) < 0.4] = 3
    if kind == 6 and v > 0:
        g[v] = g[v - 1]
        g[v][rng.integers(0, n, 2)] = rng.integers(0, 4, 2)
    if kind == 7:
        g[v] = 3
remap = np.array([3, 2, 0, 1], dtype=np.uint8)  # PgrGet code -> .bed code
b = remap[g]
b = np.concatenate([b, np.zeros((m, (-n) % 4), dtype=np.uint8)], axis=1).reshape(m, -1, 4)
by = (b[..., 0] | (b[..., 1] << 2) | (b[..., 2] << 4) | (b[..., 3] << 6)).astype(np.uint8)
open("b.bed", "wb").write(bytes([0x6C, 0x1B, 1]) + by.tobytes())
open("b.bim", "w").write("".join(f"{1 + v // 200}\tv{v}\t0\t{100 + v}\tA\tC\n" for v in range(m)))
open("b.fam", "w").write("".join(f"f{k}\ti{k}\t0\t0\t{1 + k % 2}\t-9\n" for k in range(n)))
PY
$P --bfile b --make-pgen --out $T/b --threads 1 > /dev/null
cp $T/b.pgen b_mode10.pgen; cp $T/b.pvar b.pvar; cp $T/b.psam b.psam
# --- set Q: rare-variant pre-scan accounting of the reference's KING table (NSNP), inputs from make_quirk_set.py
python make_quirk_set.py
$P --bfile q --make-king-table counts cols=+ibs1,+ibs --threads 2 --out $T/q_king > /dev/null
cp $T/q_king.kin0 q_king.kin0
$P --bfile q --make-king-table --king-table-filter -0.2 --threads 2 --out $T/q_kingp > /dev/null
cp $T/q_kingp.kin0 q_kingp.kin0
