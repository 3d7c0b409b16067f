#!/usr/bin/env Rscript
# Golden OUTPUTS of the real reference (R + Bioconductor + recoup), for machines that have them.
#
#     Rscript tools/make_r_golden.R [out_dir = tests/golden/r_outputs]
#
# R cannot be installed in the build image of this repository (no network), so the parity of
# recoup_b200 is pinned by a CPU restatement (oracle/) only: "parity unpinned".  Running this
# script once on any machine with `BiocManager::install("recoup")` closes that gap: it writes
# plain CSV files that tests/test_r_golden.py compares with the oracle (and, on a GPU box, with
# the CUDA path) -- coverage bit-exact, matrices within 1e-6 relative.
#
# Cases: the man-page examples of the hot-path functions on the bundled data
# (man/coverageRef.Rd:49-62, man/profileMatrix.Rd:32-51, man/coverageRnaRef.Rd:50-70 of the
# reference) = BASELINE.json config C1 and the reference's own smoke test
# (inst/unitTests/test_recoup.R:4-26), plus the base-R / IRanges known answers of
# tests/test_oracle_kat.py.
suppressPackageStartupMessages({
    library(recoup)
    library(GenomicRanges)
})
args <- commandArgs(trailingOnly=TRUE)
out <- if (length(args) >= 1) args[1] else file.path("tests","golden","r_outputs")
dir.create(out,recursive=TRUE,showWarnings=FALSE)

write_cov <- function(cov,file) {
    # one line per region: name, NULL flag, then the run-length encoding values:lengths
    con <- file(file,"w")
    for (n in names(cov)) {
        x <- cov[[n]]
        if (is.null(x)) {
            writeLines(paste(n,"NULL",sep=","),con)
        } else {
            r <- S4Vectors::Rle(as.integer(x))
            writeLines(paste(n,length(x),paste(S4Vectors::runValue(r),S4Vectors::runLength(r),
                sep=":",collapse=" "),sep=","),con)
        }
    }
    close(con)
}
write_mat <- function(m,file)
    write.table(format(m,digits=17),file,sep=",",quote=FALSE,col.names=FALSE)

data("recoup_test_data",package="recoup")
genes <- makeGRangesFromDataFrame(df=test.genome,keep.extra.columns=TRUE)

# ---- C1: TSS +-2 kb, 100 bins (per-sample coverage + profile) ----
inp <- coverageRef(test.input,genomeRanges=genes,region="tss",flank=c(2000,2000))
inp <- profileMatrix(inp,flank=c(2000,2000),binParams=list(flankBinSize=0,
    regionBinSize=100,sumStat="mean",interpolation="auto"),rc=NULL)
for (s in names(inp)) {
    write_cov(inp[[s]]$coverage,file.path(out,paste0("tss_",s,"_coverage.csv")))
    write_mat(inp[[s]]$profile,file.path(out,paste0("tss_",s,"_profile.csv")))
}
# ---- gene bodies + 2 kb flanks, 50 + 150 + 50 bins (test_recoup.R:15-26) ----
inp <- coverageRef(test.input,genomeRanges=genes,region="genebody",flank=c(2000,2000))
inp <- profileMatrix(inp,flank=c(2000,2000),binParams=list(flankBinSize=50,
    regionBinSize=150,sumStat="mean",interpolation="auto"),rc=NULL)
for (s in names(inp)) {
    write_cov(inp[[s]]$coverage,file.path(out,paste0("genebody_",s,"_coverage.csv")))
    write_mat(inp[[s]]$profile,file.path(out,paste0("genebody_",s,"_profile.csv")))
}
# ---- RNA: exons stitched to genes + flanks (man/coverageRnaRef.Rd) ----
inp <- coverageRnaRef(test.input,genomeRanges=test.exons,helperRanges=genes,
    flank=c(2000,2000))
inp <- profileMatrix(inp,flank=c(2000,2000),binParams=list(flankBinSize=50,
    regionBinSize=150,sumStat="mean",interpolation="auto"),rc=NULL)
for (s in names(inp)) {
    write_cov(inp[[s]]$coverage,file.path(out,paste0("rna_",s,"_coverage.csv")))
    write_mat(inp[[s]]$profile,file.path(out,paste0("rna_",s,"_profile.csv")))
}
# ---- kmeans of the C1 profiles, both samples cbind-ed (kmeansDesign, util.R:140-197) ----
inp <- coverageRef(test.input,genomeRanges=genes,region="tss",flank=c(2000,2000))
inp <- profileMatrix(inp,flank=c(2000,2000),binParams=list(flankBinSize=0,
    regionBinSize=100,sumStat="mean",interpolation="auto"),rc=NULL)
km_x <- do.call("cbind",lapply(inp,function(s) s$profile))
for (alg in c("Hartigan-Wong","Lloyd","MacQueen")) {
    for (ns in c(1,20)) {
        set.seed(42)
        km <- kmeans(km_x,centers=5,iter.max=20,nstart=ns,algorithm=alg)
        f <- file.path(out,paste0("kmeans_",gsub("-","",alg),"_nstart",ns,"_"))
        writeLines(as.character(km$cluster),paste0(f,"cluster.txt"))
        write.table(format(km$centers,digits=17),paste0(f,"centers.csv"),sep=",",quote=FALSE,
            col.names=FALSE,row.names=FALSE)
        writeLines(format(km$withinss,digits=17),paste0(f,"withinss.txt"))
        writeLines(as.character(km$iter),paste0(f,"iter.txt"))
    }
}
# ---- hclust(dist(km_x)) of the same profiles (the heat-map rows of orderBy = "hca") ----
hc <- hclust(dist(km_x))
write.table(hc$merge,file.path(out,"hclust_merge.csv"),sep=",",quote=FALSE,col.names=FALSE,
    row.names=FALSE)
writeLines(sprintf("%.17g",hc$height),file.path(out,"hclust_height.txt"))
writeLines(as.character(hc$order),file.path(out,"hclust_order.txt"))
# ---- base-R known answers ----
kat <- list()
set.seed(42); kat$sample_42_10 <- sample(1:10)
set.seed(42); kat$sample_42_100_10 <- sample(1:100,10)
for (n in c(50,100,150,200)) { set.seed(42); kat[[paste0("perm_42_",n)]] <- sample(1:n,n) }
set.seed(1); kat$runif_1 <- runif(3)
kat$spline_fmm <- spline(c(3,0,7,7,2,9,1,4,4),n=17)$y
kat$quantile7 <- unname(quantile(1:10,c(0.95,0.25,0.5)))
kat$r_version <- paste(R.version$major,R.version$minor,sep=".")
kat$sample_kind <- RNGkind()[3]
con <- file(file.path(out,"kat.txt"),"w")
for (k in names(kat)) writeLines(paste(k,paste(format(kat[[k]],digits=17),collapse=" "),sep="="),con)
close(con)
writeLines(capture.output(sessionInfo()),file.path(out,"sessionInfo.txt"))
cat("wrote",out,"\n")
