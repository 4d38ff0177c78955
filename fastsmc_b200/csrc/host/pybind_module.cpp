// pyASMC — Python bindings with the reference's class, method and keyword names
// (ref: ASMC_SRC/SRC/pybind.cpp:54-252).  Matrices are exposed as numpy arrays instead of Eigen casters.
#include <pybind11/functional.h>
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "ASMC.hpp"
#include "BinaryDataReader.hpp"
#include "CandidateOrder.hpp"
#include "Data.hpp"
#include "DecodePairsReturnStruct.hpp"
#include "DecodingParams.hpp"
#include "DecodingQuantities.hpp"
#include "FastSMC.hpp"
#include "HMM.hpp"
#include "HmmUtils.hpp"
#include "Partitioner.hpp"

namespace py = pybind11;
using namespace py::literals;

namespace
{

template <class T> py::array_t<T> matrixView(RowMajorMatrix<T>& m, py::handle owner)
{
  return py::array_t<T>({m.nRows, m.nCols}, {static_cast<long>(sizeof(T)) * m.nCols, static_cast<long>(sizeof(T))},
                        m.values.data(), owner);
}

template <class T> py::array_t<T> vectorCopy(const std::vector<T>& v, long rows, long cols)
{
  py::array_t<T> a({rows, cols});
  std::copy(v.begin(), v.end(), a.mutable_data());
  return a;
}


py::dict tablesToDict(const HMM::ModelTables& t, const DecodingQuantities& dq)
{
  py::dict d;
  const long S = t.states, L = t.sites, n = t.numDistances;
  d["initial_state_prob"] = vectorCopy(dq.initialStateProb, 1, S).attr("reshape")(S);
  d["expected_times"] = vectorCopy(dq.expectedTimes, 1, S).attr("reshape")(S);
  d["column_ratios"] = vectorCopy(dq.columnRatios, 1, S).attr("reshape")(S);
  d["emission1"] = vectorCopy(t.emission1, L, S);
  d["emission0minus1"] = vectorCopy(t.emission0minus1, L, S);
  d["emission2minus0"] = vectorCopy(t.emission2minus0, L, S);
  d["D"] = vectorCopy(t.D, n, S);
  d["B"] = vectorCopy(t.B, n, S);
  d["U"] = vectorCopy(t.U, n, S);
  d["RR"] = vectorCopy(t.RR, n, S);
  d["distance_row"] = vectorCopy(t.distanceRow, 1, L).attr("reshape")(L);
  d["state_threshold"] = t.stateThreshold;
  d["age_threshold"] = t.ageThreshold;
  d["probability_threshold"] = t.probabilityThreshold;
  return d;
}
}  // namespace

PYBIND11_MODULE(pyASMC, m)
{
  m.doc() = "fastsmc_b200: B200-native FastSMC / ASMC decoding behind the reference's pyASMC interface";

  py::enum_<DecodingModeOverall>(m, "DecodingModeOverall", py::arithmetic())
      .value("sequence", DecodingModeOverall::sequence)
      .value("array", DecodingModeOverall::array);
  py::enum_<DecodingMode>(m, "DecodingMode", py::arithmetic())
      .value("sequenceFolded", DecodingMode::sequenceFolded)
      .value("arrayFolded", DecodingMode::arrayFolded)
      .value("sequence", DecodingMode::sequence)
      .value("array", DecodingMode::array);

  py::class_<DecodingReturnValues>(m, "DecodingReturnValues")
      .def_property_readonly("sumOverPairs",
                             [](py::object self) {
                               return matrixView(self.cast<DecodingReturnValues&>().sumOverPairs, self);
                             })
      .def_property_readonly("sumOverPairs00",
                             [](py::object self) {
                               return matrixView(self.cast<DecodingReturnValues&>().sumOverPairs00, self);
                             })
      .def_property_readonly("sumOverPairs01",
                             [](py::object self) {
                               return matrixView(self.cast<DecodingReturnValues&>().sumOverPairs01, self);
                             })
      .def_property_readonly("sumOverPairs11",
                             [](py::object self) {
                               return matrixView(self.cast<DecodingReturnValues&>().sumOverPairs11, self);
                             })
      .def_readwrite("sites", &DecodingReturnValues::sites)
      .def_readwrite("states", &DecodingReturnValues::states)
      .def_readwrite("siteWasFlippedDuringFolding", &DecodingReturnValues::siteWasFlippedDuringFolding);

  py::class_<DecodePairsReturnStruct>(m, "DecodePairsReturnStruct")
      .def_readwrite("per_pair_indices", &DecodePairsReturnStruct::perPairIndices)
      .def_property_readonly("per_pair_posterior_means",
                             [](py::object self) {
                               auto& s = self.cast<DecodePairsReturnStruct&>();
                               return matrixView(s.perPairPosteriorMeans, self);
                             })
      .def_property_readonly("per_pair_MAPs",
                             [](py::object self) {
                               auto& s = self.cast<DecodePairsReturnStruct&>();
                               return matrixView(s.perPairMAPs, self);
                             })
      .def_property_readonly("sum_of_posteriors",
                             [](py::object self) {
                               auto& s = self.cast<DecodePairsReturnStruct&>();
                               return matrixView(s.sumOfPosteriors, self);
                             })
      .def_property_readonly("per_pair_posteriors",
                             [](py::object self) {
                               auto& s = self.cast<DecodePairsReturnStruct&>();
                               py::list out;
                               for (auto& mat : s.perPairPosteriors) {
                                 out.append(matrixView(mat, self));
                               }
                               return out;
                             })
      .def_readwrite("min_posterior_means", &DecodePairsReturnStruct::minPosteriorMeans)
      .def_readwrite("argmin_posterior_means", &DecodePairsReturnStruct::argminPosteriorMeans)
      .def_readwrite("min_MAPs", &DecodePairsReturnStruct::minMAPs)
      .def_readwrite("argmin_MAPs", &DecodePairsReturnStruct::argminMAPs);

  py::class_<Individual>(m, "Individual")
      .def(py::init<int>(), "numOfSites"_a = 0)
      .def("setGenotype", &Individual::setGenotype, "hap"_a, "pos"_a, "val"_a)
      .def_readwrite("genotype1", &Individual::genotype1)
      .def_readwrite("genotype2", &Individual::genotype2);

  py::class_<PairObservations>(m, "PairObservations")
      .def_readwrite("obsBits", &PairObservations::obsBits)
      .def_readwrite("homMinorBits", &PairObservations::homMinorBits)
      .def_readwrite("iHap", &PairObservations::iHap)
      .def_readwrite("jHap", &PairObservations::jHap)
      .def_readwrite("iInd", &PairObservations::iInd)
      .def_readwrite("jInd", &PairObservations::jInd);

  py::class_<DecodingQuantities>(m, "DecodingQuantities")
      .def(py::init<const std::string&>())
      .def_readwrite("CSFSSamples", &DecodingQuantities::CSFSSamples)
      .def_readwrite("states", &DecodingQuantities::states)
      .def_readwrite("initialStateProb", &DecodingQuantities::initialStateProb)
      .def_readwrite("expectedTimes", &DecodingQuantities::expectedTimes)
      .def_readwrite("discretization", &DecodingQuantities::discretization)
      .def_readwrite("timeVector", &DecodingQuantities::timeVector)
      .def_readwrite("columnRatios", &DecodingQuantities::columnRatios)
      .def_readwrite("classicEmissionTable", &DecodingQuantities::classicEmissionTable)
      .def_readwrite("compressedEmissionTable", &DecodingQuantities::compressedEmissionTable)
      .def_readwrite("Dvectors", &DecodingQuantities::Dvectors)
      .def_readwrite("Bvectors", &DecodingQuantities::Bvectors)
      .def_readwrite("Uvectors", &DecodingQuantities::Uvectors)
      .def_readwrite("rowRatioVectors", &DecodingQuantities::rowRatioVectors)
      .def_readwrite("homozygousEmissionMap", &DecodingQuantities::homozygousEmissionMap)
      .def_readwrite("CSFSmap", &DecodingQuantities::CSFSmap)
      .def_readwrite("foldedCSFSmap", &DecodingQuantities::foldedCSFSmap)
      .def_readwrite("ascertainedCSFSmap", &DecodingQuantities::ascertainedCSFSmap)
      .def_readwrite("foldedAscertainedCSFSmap", &DecodingQuantities::foldedAscertainedCSFSmap);

  py::class_<DecodingParams>(m, "DecodingParams")
      .def(py::init<std::string, std::string, std::string, int, int, std::string, bool, bool, bool, bool, float, bool,
                    bool, bool, std::string, bool, bool>(),
           "inFileRoot"_a, "decodingQuantFile"_a, "outFileRoot"_a = "", "jobs"_a = 1, "jobInd"_a = 1,
           "decodingModeString"_a = "array", "decodingSequence"_a = false, "usingCSFS"_a = true, "compress"_a = false,
           "useAncestral"_a = false, "skipCSFSdistance"_a = 0.f, "noBatches"_a = false, "doPosteriorSums"_a = false,
           "doPerPairPosteriorMean"_a = false, "expectedCoalTimesFile"_a = "", "withinOnly"_a = false,
           "doMajorMinorPosteriorSums"_a = false)
      .def(py::init<>())
      .def(py::init<std::string, std::string, std::string, bool>(), "in_dir"_a, "decoding_quants"_a, "out_dir"_a,
           "FastSMC"_a = true)
      .def("validateParamsFastSMC", &DecodingParams::validateParamsFastSMC)
      .def_readwrite("inFileRoot", &DecodingParams::inFileRoot)
      .def_readwrite("decodingQuantFile", &DecodingParams::decodingQuantFile)
      .def_readwrite("outFileRoot", &DecodingParams::outFileRoot)
      .def_readwrite("jobs", &DecodingParams::jobs)
      .def_readwrite("jobInd", &DecodingParams::jobInd)
      .def_readwrite("decodingModeString", &DecodingParams::decodingModeString)
      .def_readwrite("decodingMode", &DecodingParams::decodingMode)
      .def_readwrite("decodingSequence", &DecodingParams::decodingSequence)
      .def_readwrite("foldData", &DecodingParams::foldData)
      .def_readwrite("usingCSFS", &DecodingParams::usingCSFS)
      .def_readwrite("compress", &DecodingParams::compress)
      .def_readwrite("useAncestral", &DecodingParams::useAncestral)
      .def_readwrite("skipCSFSdistance", &DecodingParams::skipCSFSdistance)
      .def_readwrite("noBatches", &DecodingParams::noBatches)
      .def_readwrite("batchSize", &DecodingParams::batchSize)
      .def_readwrite("recallThreshold", &DecodingParams::recallThreshold)
      .def_readwrite("skip", &DecodingParams::skip)
      .def_readwrite("gap", &DecodingParams::gap)
      .def_readwrite("max_seeds", &DecodingParams::max_seeds)
      .def_readwrite("min_maf", &DecodingParams::min_maf)
      .def_readwrite("min_m", &DecodingParams::min_m)
      .def_readwrite("hashing", &DecodingParams::hashing)
      .def_readwrite("FastSMC", &DecodingParams::FastSMC)
      .def_readwrite("BIN_OUT", &DecodingParams::BIN_OUT)
      .def_readwrite("useKnownSeed", &DecodingParams::useKnownSeed)
      .def_readwrite("outputIbdSegmentLength", &DecodingParams::outputIbdSegmentLength)
      .def_readwrite("hashingWordSize", &DecodingParams::hashingWordSize)
      .def_readwrite("constReadAhead", &DecodingParams::constReadAhead)
      .def_readwrite("haploid", &DecodingParams::haploid)
      .def_readwrite("time", &DecodingParams::time)
      .def_readwrite("noConditionalAgeEstimates", &DecodingParams::noConditionalAgeEstimates)
      .def_readwrite("doPosteriorSums", &DecodingParams::doPosteriorSums)
      .def_readwrite("doPerPairMAP", &DecodingParams::doPerPairMAP)
      .def_readwrite("doPerPairPosteriorMean", &DecodingParams::doPerPairPosteriorMean)
      .def_readwrite("expectedCoalTimesFile", &DecodingParams::expectedCoalTimesFile)
      .def_readwrite("withinOnly", &DecodingParams::withinOnly)
      .def_readwrite("doMajorMinorPosteriorSums", &DecodingParams::doMajorMinorPosteriorSums)
      // B200 build
      .def_readwrite("device", &DecodingParams::device)
      .def_readwrite("exactArithmetic", &DecodingParams::exactArithmetic)
      .def_readwrite("referenceCandidateOrder", &DecodingParams::referenceCandidateOrder)
      .def_readwrite("hapBitCache", &DecodingParams::hapBitCache)
      .def_readwrite("outputCompressionLevel", &DecodingParams::outputCompressionLevel)
      .def_readwrite("outputThreads", &DecodingParams::outputThreads)
      .def_readwrite("verbose", &DecodingParams::verbose);

  py::class_<IbdPairDataLine>(m, "IbdPairDataLine")
      .def(py::init<>())
      .def_readwrite("ind1FamId", &IbdPairDataLine::ind1FamId)
      .def_readwrite("ind1Id", &IbdPairDataLine::ind1Id)
      .def_readwrite("ind1Hap", &IbdPairDataLine::ind1Hap)
      .def_readwrite("ind2FamId", &IbdPairDataLine::ind2FamId)
      .def_readwrite("ind2Id", &IbdPairDataLine::ind2Id)
      .def_readwrite("ind2Hap", &IbdPairDataLine::ind2Hap)
      .def_readwrite("chromosome", &IbdPairDataLine::chromosome)
      .def_readwrite("ibdStart", &IbdPairDataLine::ibdStart)
      .def_readwrite("ibdEnd", &IbdPairDataLine::ibdEnd)
      .def_readwrite("lengthInCentimorgans", &IbdPairDataLine::lengthInCentimorgans)
      .def_readwrite("ibdScore", &IbdPairDataLine::ibdScore)
      .def_readwrite("postEst", &IbdPairDataLine::postEst)
      .def_readwrite("mapEst", &IbdPairDataLine::mapEst)
      .def("toString", &IbdPairDataLine::toString);

  py::class_<BinaryDataReader>(m, "BinaryDataReader")
      .def(py::init<const std::string&>(), "binaryFile"_a)
      .def("getNextLine", &BinaryDataReader::getNextLine)
      .def("moreLinesInFile", &BinaryDataReader::moreLinesInFile);

  py::class_<Data>(m, "Data")
      .def(py::init<const DecodingParams&>(), "params"_a)
      .def_static("forJob", &Data::forJob, "whole"_a, "params"_a)
      .def_static("countHapLines", &Data::countHapLines)
      .def_static("countSamplesLines", &Data::countSamplesLines)
      .def_static(
          "fromArrays",
          [](const DecodingParams& p, const std::vector<std::string>& fam, const std::vector<std::string>& iid,
             py::array_t<uint8_t, py::array::c_style | py::array::forcecast> raw, const std::vector<int>& bp,
             const std::vector<double>& cM, int chr) {
            if (raw.ndim() != 2) {
              throw std::runtime_error("rawAlleles must be [numHaps][sites]");
            }
            return Data::fromArrays(p, fam, iid, raw.data(), raw.shape(0), static_cast<int>(raw.shape(1)), bp, cM, chr);
          },
          "params"_a, "famIds"_a, "iids"_a, "rawAlleles"_a, "physicalPositions"_a, "centimorgans"_a, "chromosome"_a)
      .def_readwrite("FamIDList", &Data::FamIDList)
      .def_readwrite("IIDList", &Data::IIDList)
      .def_readwrite("famAndIndNameList", &Data::famAndIndNameList)
      .def_property_readonly("individuals",
                             [](const Data& d) {
                               std::vector<Individual> v;
                               for (unsigned long i = 0; i < d.numLoadedIndividuals(); ++i) {
                                 v.push_back(d.individual(i));
                               }
                               return v;
                             })
      .def_readwrite("sampleSize", &Data::sampleSize)
      .def_readwrite("haploidSampleSize", &Data::haploidSampleSize)
      .def_readwrite("sites", &Data::sites)
      .def_readwrite("decodingUsesCSFS", &Data::decodingUsesCSFS)
      .def_readwrite("geneticPositions", &Data::geneticPositions)
      .def_readwrite("physicalPositions", &Data::physicalPositions)
      .def_readwrite("siteWasFlippedDuringFolding", &Data::siteWasFlippedDuringFolding)
      .def_readwrite("recRateAtMarker", &Data::recRateAtMarker)
      .def_readwrite("chrNumber", &Data::chrNumber)
      .def_readwrite("windowSize", &Data::windowSize)
      .def_readwrite("w_i", &Data::w_i)
      .def_readwrite("w_j", &Data::w_j)
      .def_readwrite("is_j_above_diag", &Data::is_j_above_diag)
      .def_readwrite("globalHapId", &Data::globalHapId)
      .def_readonly("flipMask", &Data::flipMask)
      .def_readonly("totalSamplesCount", &Data::totalSamplesCount)
      .def_readonly("derivedAlleleCounts", &Data::derivedAlleleCounts)
      .def_readwrite("wordsPerHap", &Data::wordsPerHap)
      .def_property_readonly("hapBits",
                             [](const Data& d) {
                               return vectorCopy(d.hapBits, static_cast<long>(d.numLoadedHaplotypes()), d.wordsPerHap);
                             })
      .def("calculateUndistinguishedCounts", &Data::calculateUndistinguishedCounts);

  py::class_<HMM::RunStats>(m, "RunStats")
      .def_readonly("pairsDecoded", &HMM::RunStats::pairsDecoded)
      .def_readonly("batches", &HMM::RunStats::batches)
      .def_readonly("segments", &HMM::RunStats::segments)
      .def_readonly("decodeCalls", &HMM::RunStats::decodeCalls)
      .def_readonly("pairSites", &HMM::RunStats::pairSites)
      .def_readonly("kernelMs", &HMM::RunStats::kernelMs)
      .def_readonly("deviceMs", &HMM::RunStats::deviceMs)
      .def_readonly("decodeWallS", &HMM::RunStats::decodeWallS)
      .def_readonly("outputWallS", &HMM::RunStats::outputWallS)
      .def_readonly("d2hBytes", &HMM::RunStats::d2hBytes);

  py::class_<HMM>(m, "HMM")
      .def(py::init([](const Data& d, const DecodingParams& p, int skip) { return new HMM(d, p, skip); }), "data"_a,
           "params"_a, "scalingSkip"_a = 1)
      .def("decode", py::overload_cast<const PairObservations&>(&HMM::decode))
      .def("decode", py::overload_cast<const PairObservations&, unsigned, unsigned>(&HMM::decode))
      .def("decodeAll", &HMM::decodeAll)
      .def("decodeSummarize", &HMM::decodeSummarize)
      .def("getDecodingReturnValues", &HMM::getDecodingReturnValues)
      .def("decodePair", &HMM::decodePair)
      .def("decodePairs", &HMM::decodePairs)
      .def("decodeFromHashing", &HMM::decodeFromHashing)
      .def("finishFromHashing", &HMM::finishFromHashing)
      .def("getBatchBuffer", &HMM::getBatchBuffer)
      .def("finishDecoding", &HMM::finishDecoding)
      .def("closeIBDFile", &HMM::closeIBDFile)
      .def("getStateThreshold", &HMM::getStateThreshold)
      .def("getDecodingQuantities", &HMM::getDecodingQuantities, py::return_value_policy::reference_internal)
      .def("makePairObs", &HMM::makePairObs, "iHap"_a, "ind1"_a, "jHap"_a, "ind2"_a, "materialise"_a = true)
      .def("getRunStats", &HMM::getRunStats, py::return_value_policy::reference_internal)
      .def("getNumberOfDetectedSegments", &HMM::getNumberOfDetectedSegments)
      .def("getDevice", &HMM::getDevice)
      .def("getModelTables", [](const HMM& h) { return tablesToDict(h.getModelTables(), h.getDecodingQuantities()); });



  py::class_<fsmc_seed_stats>(m, "SeedDeviceStats")
      .def_readonly("numMatches", &fsmc_seed_stats::numMatches)
      .def_readonly("pairVisits", &fsmc_seed_stats::pairVisits)
      .def_readonly("numStarts", &fsmc_seed_stats::numStarts)
      .def_readonly("numWords", &fsmc_seed_stats::numWords)
      .def_readonly("kernelLaunches", &fsmc_seed_stats::kernelLaunches)
      .def_readonly("kernelMs", &fsmc_seed_stats::kernelMs)
      .def_readonly("bytesRead", &fsmc_seed_stats::bytesRead)
      .def_readonly("numIntervals", &fsmc_seed_stats::numIntervals)
      .def_readonly("maxLiveNodes", &fsmc_seed_stats::maxLiveNodes)
      .def_readonly("orderEpochs", &fsmc_seed_stats::orderEpochs)
      .def_readonly("orderMs", &fsmc_seed_stats::orderMs)
      .def_readonly("rankHostMs", &fsmc_seed_stats::rankHostMs);
  py::class_<ASMC::FastSMC::SeedingStats>(m, "SeedingStats")
      .def_readonly("device", &ASMC::FastSMC::SeedingStats::device)
      .def_readonly("seedWallS", &ASMC::FastSMC::SeedingStats::seedWallS)
      .def_readonly("orderWallS", &ASMC::FastSMC::SeedingStats::orderWallS)
      .def_readonly("submitWallS", &ASMC::FastSMC::SeedingStats::submitWallS)
      .def_readonly("candidates", &ASMC::FastSMC::SeedingStats::candidates);

  py::class_<ASMC::FastSMC>(m, "FastSMC")
      .def(py::init<DecodingParams>(), "decodingParams"_a)
      .def(py::init<const std::string&, const std::string&>(), "in_dir"_a, "out_dir"_a)
      .def(py::init<DecodingParams, Data>(), "decodingParams"_a, "data"_a)
      .def("run", &ASMC::FastSMC::run, py::call_guard<py::gil_scoped_release>())
      .def("getSeedingStats", &ASMC::FastSMC::getSeedingStats, py::return_value_policy::reference_internal)
      .def("setKeepCandidates", &ASMC::FastSMC::setKeepCandidates)
      .def("getCandidates",
           [](const ASMC::FastSMC& f) {
             const auto& c = f.getCandidates();
             py::array_t<uint32_t> a({static_cast<long>(c.size()), 4l});
             auto* p = a.mutable_data();
             for (size_t i = 0; i < c.size(); ++i) {
               p[4 * i] = c[i].hapA;
               p[4 * i + 1] = c[i].hapB;
               p[4 * i + 2] = static_cast<uint32_t>(c[i].startWord);
               p[4 * i + 3] = static_cast<uint32_t>(c[i].endWord);
             }
             return a;
           })
      .def("hmm", &ASMC::FastSMC::hmm, py::return_value_policy::reference_internal)
      .def("data", &ASMC::FastSMC::data, py::return_value_policy::reference_internal)
      .def("getRunWallSeconds", &ASMC::FastSMC::getRunWallSeconds);

  py::class_<ASMC::ASMC>(m, "ASMC")
      .def(py::init<DecodingParams>(), "decodingParams"_a)
      .def(py::init<const std::string&, const std::string&, const std::string&>(), "in_dir"_a, "decoding_quants"_a,
           "out_dir"_a = "")
      .def("decodeAllInJob", &ASMC::ASMC::decodeAllInJob)
      .def("decodePairs",
           py::overload_cast<const std::vector<unsigned long>&, const std::vector<unsigned long>&, bool, bool, bool, bool>(
               &ASMC::ASMC::decodePairs),
           "hap_indices_a"_a, "hap_indices_b"_a, "per_pair_posteriors"_a = false, "sum_of_posteriors"_a = false,
           "per_pair_posterior_means"_a = false, "per_pair_MAPs"_a = false)
      .def("decodePairs",
           py::overload_cast<const std::vector<std::string>&, const std::vector<std::string>&, bool, bool, bool, bool>(
               &ASMC::ASMC::decodePairs),
           "hap_ids_a"_a, "hap_ids_b"_a, "per_pair_posteriors"_a = false, "sum_of_posteriors"_a = false,
           "per_pair_posterior_means"_a = false, "per_pair_MAPs"_a = false)
      // device-resident outputs: raw device pointers (e.g. torch's data_ptr()) and a cudaStream_t as integers, 0 = none;
      // returns per_pair_indices.  fastsmc_b200.cuda_results.decode_pairs_cuda allocates and checks the tensors.
      .def("decodePairsToDevice",
           [](ASMC::ASMC& self, const py::object& a, const py::object& b, const uintptr_t perPairPosteriors,
              const uintptr_t sumOfPosteriors, const uintptr_t perPairPosteriorMeans, const uintptr_t perPairMAPs,
              const uintptr_t stream) {
             HMM::DeviceOutputs out;
             out.perPairPosteriors = reinterpret_cast<float*>(perPairPosteriors);
             out.sumOfPosteriors = reinterpret_cast<float*>(sumOfPosteriors);
             out.perPairPosteriorMeans = reinterpret_cast<float*>(perPairPosteriorMeans);
             out.perPairMAPs = reinterpret_cast<int32_t*>(perPairMAPs);
             out.stream = reinterpret_cast<void*>(stream);
             const py::list la(a), lb(b);
             if (la.size() > 0 && py::isinstance<py::str>(la[0])) {
               const auto ia = la.cast<std::vector<std::string>>(), ib = lb.cast<std::vector<std::string>>();
               py::gil_scoped_release release;
               return self.decodePairsToDevice(ia, ib, out);
             }
             const auto ia = la.cast<std::vector<unsigned long>>(), ib = lb.cast<std::vector<unsigned long>>();
             py::gil_scoped_release release;
             return self.decodePairsToDevice(ia, ib, out);
           },
           "haps_a"_a, "haps_b"_a, "per_pair_posteriors"_a = 0, "sum_of_posteriors"_a = 0, "per_pair_posterior_means"_a = 0,
           "per_pair_MAPs"_a = 0, "stream"_a = 0)
      .def("get_copy_of_results", &ASMC::ASMC::getCopyOfResults, py::return_value_policy::copy)
      .def("get_ref_of_results", &ASMC::ASMC::getRefOfResults, py::return_value_policy::reference_internal)
      .def("hmm", &ASMC::ASMC::hmm, py::return_value_policy::reference_internal);


  // multi-GPU: the jobs of one data set dealt to the GPUs of the box (no collective; ref: FastSMC_example_multiple_jobs.sh)
  py::class_<ASMC::JobReport>(m, "JobReport")
      .def_readonly("jobInd", &ASMC::JobReport::jobInd)
      .def_readonly("device", &ASMC::JobReport::device)
      .def_readonly("candidates", &ASMC::JobReport::candidates)
      .def_readonly("pairsDecoded", &ASMC::JobReport::pairsDecoded)
      .def_readonly("segments", &ASMC::JobReport::segments)
      .def_readonly("pairSites", &ASMC::JobReport::pairSites)
      .def_readonly("kernelMs", &ASMC::JobReport::kernelMs)
      .def_readonly("seedMs", &ASMC::JobReport::seedMs)
      .def_readonly("wallSeconds", &ASMC::JobReport::wallSeconds)
      .def_readonly("prepareSeconds", &ASMC::JobReport::prepareSeconds)
      .def_readonly("cutSeconds", &ASMC::JobReport::cutSeconds)
      .def_readonly("tablesSeconds", &ASMC::JobReport::tablesSeconds)
      .def_readonly("uploadSeconds", &ASMC::JobReport::uploadSeconds)
      .def_readonly("seedSeconds", &ASMC::JobReport::seedSeconds)
      .def_readonly("orderSeconds", &ASMC::JobReport::orderSeconds)
      .def_readonly("decodeSeconds", &ASMC::JobReport::decodeSeconds)
      .def_readonly("outputSeconds", &ASMC::JobReport::outputSeconds)
      .def_readonly("error", &ASMC::JobReport::error);
  m.def("jobOrder", &ASMC::jobOrder, "jobs"_a);
  m.def("jobsOfRank", &ASMC::jobsOfRank, "jobs"_a, "world"_a, "rank"_a);
  m.def("runAllJobs", &ASMC::runAllJobs, "params"_a, "devices"_a, py::call_guard<py::gil_scoped_release>());
  // the job source is a Python callable (e.g. a counter shared by torchrun ranks); pybind re-acquires the GIL to call it
  m.def("runJobs", &ASMC::runJobs, "params"_a, "whole"_a, "nextJob"_a, "devices"_a, py::call_guard<py::gil_scoped_release>());

  // host-only pieces, callable without a GPU (used by the CPU test-suite)
  m.def(
      "prepareModelTables",
      [](const Data& data, const DecodingParams& params) {
        const DecodingQuantities dq(params.decodingQuantFile);
        return tablesToDict(HMM::buildModelTables(data, dq, params), dq);
      },
      "data"_a, "params"_a);
  m.def(
      "seedGroupRanks",
      [](const Data& data, const int maxSeeds, const int readAhead) {
        const uint32_t H = static_cast<uint32_t>(data.numLoadedHaplotypes());
        const int W = data.sites / 64;
        auto rawWord = [&](uint32_t h, int w) {
          return data.hapBits[static_cast<size_t>(h) * data.wordsPerHap + w] ^ data.flipMask[w];
        };
        const std::vector<uint32_t> r = candidate_order::seedGroupRanks(H, W, rawWord, 0, maxSeeds, readAhead);
        py::array_t<uint32_t> out({static_cast<py::ssize_t>(W), static_cast<py::ssize_t>(H)});
        std::copy(r.begin(), r.end(), out.mutable_data());
        return out;
      },
      "data"_a, "max_seeds"_a = 0, "read_ahead"_a = 10);
  m.def(
      "replayReferenceOrder",
      [](py::array_t<int64_t, py::array::c_style | py::array::forcecast> intervals, const Data& data, int gap,
         float min_m, bool fast) {
        std::vector<fsmc_match> iv(intervals.shape(0));
        for (long i = 0; i < intervals.shape(0); ++i) {
          iv[i] = fsmc_match{static_cast<uint32_t>(intervals.at(i, 0)), static_cast<uint32_t>(intervals.at(i, 1)),
                             static_cast<int32_t>(intervals.at(i, 2)), static_cast<int32_t>(intervals.at(i, 3))};
        }
        std::vector<int64_t> order;
        auto rawWord = [&](uint32_t h, int w) {
          return data.hapBits[static_cast<size_t>(h) * data.wordsPerHap + w] ^ data.flipMask[w];
        };
        auto longEnough = [&](const fsmc_match& x) {
          return asmc::cmBetween(x.startWord, x.endWord, data.geneticPositions, 64) >= static_cast<double>(min_m);
        };
        auto emit = [&](int64_t i) { order.push_back(i); };
        if (fast) {
          candidate_order::replayReferenceOrderFast(iv, static_cast<uint32_t>(data.numLoadedHaplotypes()), data.sites / 64,
                                                    gap, rawWord, longEnough, emit);
        } else {
          candidate_order::replayReferenceOrder(iv, static_cast<uint32_t>(data.numLoadedHaplotypes()), data.sites / 64, gap,
                                                rawWord, longEnough, emit);
        }
        return order;
      },
      "intervals"_a, "data"_a, "gap"_a, "min_m"_a, "fast"_a = true);

  // helpers with reference known-answer tests (ref: ASMC_SRC/TESTS/test_hmm_utils.cpp, test_hashing.cpp)
  m.def("roundMorgans", &asmc::roundMorgans, "value"_a, "precision"_a, "min"_a);
  m.def("roundPhysical", &asmc::roundPhysical, "value"_a, "precision"_a);
  m.def("getFromPosition", &asmc::getFromPosition, "geneticPositions"_a, "from"_a, "cmDist"_a = 0.5f);
  m.def("getToPosition", &asmc::getToPosition, "geneticPositions"_a, "to"_a, "cmDist"_a = 0.5f);
  m.def("cmBetween", &asmc::cmBetween, "w1"_a, "w2"_a, "geneticPositions"_a, "wordSize"_a);
  m.def("hapToDipId", &asmc::hapToDipId);
  m.def("dipToHapId", &asmc::dipToHapId);
  m.def("indPlusHapToCombinedId", &asmc::indPlusHapToCombinedId);
  m.def("combinedIdToIndPlusHap", &asmc::combinedIdToIndPlusHap);
  m.def("getIndIdxFromIdString", &asmc::getIndIdxFromIdString);
}
