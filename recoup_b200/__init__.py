"""recoup_b200 -- B200-native (sm_100a CUDA) implementation of recoup's coverage -> profile
matrix hot path behind the reference's own R-level interface (see DESIGN.md / INTEGRATION.md).

Public names mirror /root/reference/NAMESPACE:17-19,25 and the internal closures those call.
Importing requires recoup_b200/librecoup_b200.so (built by __graft_entry__.build()); every
compute call requires a B200 -- there is no CPU fallback.
"""
from . import _lib
from ._lib import RecoupError, init, set_coverage_path, shutdown
from .consumers import (NamedVector, calcDesignPlotProfiles, calcPlotProfiles, colProfile, groupColProfile, hclust,
                        heatmapClusters, heatmapScale, kmeans, kmeansDesign, matrixQuantile, orderProfiles, rowStat,
                        sortIndex)
from .coverage import (CoverageList, DeviceReads, calcCoverage, coverageRef, coverageRnaRef,
                       device_reads, set_verbose)
from .preprocess import SelectedGRanges, preprocessRanges, readRanges, sampleSorted, widthQuantile
from .profile import (ProfileMatrix, baseCoverageMatrix, binCoverageMatrix, coverageProfile,
                      haveEqualLengths, profileMatrix)
from .readers import (BigWigTrack, DecodedGRanges, ScanBamParam, decodeBam, readBam, readBed, readBigWig,
                      readRangesFile, scanBamFlag)
from .ranges import GRanges, GRangesList, Rle, getFlankingRanges, getRegionalRanges

__all__ = [
    "RecoupError", "init", "shutdown", "set_coverage_path", "GRanges", "GRangesList", "Rle",
    "getRegionalRanges", "getFlankingRanges", "calcCoverage", "coverageRef", "coverageRnaRef", "CoverageList",
    "DeviceReads", "device_reads", "profileMatrix", "binCoverageMatrix", "baseCoverageMatrix",
    "haveEqualLengths", "coverageProfile", "ProfileMatrix", "set_verbose", "calcPlotProfiles", "orderProfiles",
    "heatmapScale", "colProfile", "rowStat", "sortIndex", "matrixQuantile", "preprocessRanges",
    "readRanges", "SelectedGRanges", "sampleSorted", "widthQuantile", "readBam", "readBed", "readRangesFile",
    "decodeBam", "DecodedGRanges", "ScanBamParam", "scanBamFlag", "readBigWig", "BigWigTrack",
    "kmeans", "kmeansDesign", "NamedVector", "hclust", "heatmapClusters", "calcDesignPlotProfiles",
    "groupColProfile",
]
