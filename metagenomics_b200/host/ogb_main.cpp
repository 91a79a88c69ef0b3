// ogb_main.cpp -- the reference's main() (MetaGenomics/main.cpp:23-51) up to the end of the
// overlap-graph build, written against the drop-in classes of this directory. The call site is
// character-for-character the reference's (main.cpp:33,45-47); everything after it in the reference
// (calculateFlow, the three simplification loops, printGraph) is host code that consumes the graph
// this program produces and is not part of this library.
//
//   ogb_overlap -l minOverlap [-se n files...] [-pe n files...] [-f prefix] [--dump file] [--unitigs file] [--coverage file]
//               [--samples n files... --depths file [--mismatches d] [--sam dir]]
//
// --dump writes the graph in the binary format the parity tests read, so one comparator reads
// the output of the unmodified reference and of this program. --unitigs writes the sequences of the canonical unitigs of the
// simplified graph as FASTA, spelled on the device (OverlapGraph::spellInBuild, saveUnitigsToFile). --coverage writes their per-base
// read depth summary as TSV, contained reads included (saveUnitigCoverageToFile); the names join with the FASTA's. --samples with
// --depths maps the reads of every sample file onto the unitigs and writes the contig x sample depth table binners take, in MetaBAT's
// layout, one column pair per sample named after the file's basename (saveSampleDepthsToFile); --mismatches lets every read count
// with up to d substitutions (at most floor(L / K) - 1 for a read of length L, K = min(32, minOverlap + 1)). --sam also writes the
// placements of every sample's reads as SAM, dir/<basename of the sample file>.sam, with the file's read names (the directory is
// created if missing).
#include "Common.h"
#include "Dataset.h"
#include "Edge.h"
#include "HashTable.h"
#include "OverlapGraph.h"

#include <cerrno>
#include <cstring>
#include <set>
#include <sys/stat.h>

static unsigned long long fnv1a(const string &s)
{
	unsigned long long h = 1469598103934665603ULL;
	for (size_t i = 0; i < s.size(); i++) { h ^= (unsigned char)s[i]; h *= 1099511628211ULL; }
	return h;
}
template <class T> static void put(FILE *f, T v) { fwrite(&v, sizeof(T), 1, f); }

static void dumpGraph(const char *path, Dataset *dataSet, OverlapGraph *overlapGraph, UINT64 minimumOverlapLength)
{
	FILE *f = fopen(path, "wb");
	if (!f) throw OgbFailure(OGB_E_IO, string("Unable to open file: ") + path);
	vector<vector<Edge *> *> *graph = overlapGraph->getGraph();
	UINT64 n = dataSet->getNumberOfUniqueReads(), nEdges = 0;
	for (UINT64 i = 1; i < graph->size(); i++) nEdges += graph->at(i)->size();
	put<unsigned long long>(f, 0x31504d554442474fULL);
	put<unsigned long long>(f, n);
	put<unsigned long long>(f, nEdges);
	put<unsigned long long>(f, overlapGraph->getNumberOfNodes());
	put<unsigned long long>(f, overlapGraph->getNumberOfEdges());
	put<unsigned long long>(f, minimumOverlapLength - 1);
	for (UINT64 i = 1; i <= n; i++) {
		Read *r = dataSet->getReadFromID(i);
		put<unsigned long long>(f, r->superReadID);
		put<unsigned int>(f, (unsigned int)r->getReadLength());
		put<unsigned int>(f, (unsigned int)r->getFrequency());
		put<unsigned long long>(f, fnv1a(r->getStringForward()));
	}
	for (UINT64 i = 1; i < graph->size(); i++)
		for (UINT64 k = 0; k < graph->at(i)->size(); k++) {
			Edge *e = graph->at(i)->at(k);
			if (e->getReverseEdge() == NULL || e->getReverseEdge()->getReverseEdge() != e) throw OgbFailure(OGB_E_STATE, "twin pointers are not linked");
			put<unsigned int>(f, (unsigned int)e->getSourceRead()->getReadNumber());
			put<unsigned int>(f, (unsigned int)e->getDestinationRead()->getReadNumber());
			put<unsigned int>(f, (unsigned int)e->getOverlapOffset());
			put<unsigned int>(f, (unsigned int)e->getOrientation());
		}
	fclose(f);
}

// every read's mate-pair list, in list order: u64 magic, u64 n, per read u32 count + count x (u32 matePairID, u32 orientation, u32 dataset) -- the format the parity tests read
static void dumpMates(const char *path, Dataset *dataSet)
{
	FILE *f = fopen(path, "wb");
	if (!f) throw OgbFailure(OGB_E_IO, string("cannot open ") + path);
	unsigned long long magic = 0x31534554414d474fULL, n = dataSet->getNumberOfUniqueReads();
	fwrite(&magic, 8, 1, f); fwrite(&n, 8, 1, f);
	for (UINT64 i = 1; i <= n; i++) {
		vector<MPlist> *l = dataSet->getReadFromID(i)->getMatePairList();
		unsigned int c = (unsigned int)l->size();
		fwrite(&c, 4, 1, f);
		for (size_t k = 0; k < l->size(); k++) {
			unsigned int v[3] = {(unsigned int)l->at(k).matePairID, (unsigned int)l->at(k).matePairOrientation, (unsigned int)l->at(k).datasetNumber};
			fwrite(v, 4, 3, f);
		}
	}
	fclose(f);
}

int main(int argc, char **argv)
{
	UINT64 minimumOverlapLength = 0;
	vector<string> pairedEndFileNames, singleEndFileNames, sampleFileNames;
	string allFileName = "";
	const char *dumpPath = NULL, *resavePath = NULL, *matesPath = NULL, *unitigsPath = NULL, *coveragePath = NULL, *depthsPath = NULL, *samDir = NULL;
	bool haveSamples = false;
	int maxMismatches = -1;																			// -1: no --mismatches
	bool startFromUnitigGraph = false;
	for (int i = 1; i < argc; i++) {
		string a = argv[i];
		if ((a == "-pe" || a == "-se") && i + 1 < argc) {
			int count = atoi(argv[++i]);
			for (int k = 0; k < count && i + 1 < argc; k++) (a == "-pe" ? pairedEndFileNames : singleEndFileNames).push_back(argv[++i]);
		} else if (a == "-f" && i + 1 < argc) allFileName = argv[++i];
		else if (a == "-l" && i + 1 < argc) minimumOverlapLength = atoi(argv[++i]);
		else if (a == "--dump" && i + 1 < argc) dumpPath = argv[++i];
		else if (a == "-s") startFromUnitigGraph = true;												// main.cpp: resume from <prefix>.unitig
		else if (a == "--resave" && i + 1 < argc) resavePath = argv[++i];
		else if (a == "--mates" && i + 1 < argc) matesPath = argv[++i];
		else if (a == "--unitigs" && i + 1 < argc) unitigsPath = argv[++i];
		else if (a == "--coverage" && i + 1 < argc) coveragePath = argv[++i];
		else if (a == "--samples" && i + 1 < argc) {
			int count = atoi(argv[++i]);
			for (int k = 0; k < count && i + 1 < argc; k++) sampleFileNames.push_back(argv[++i]);
			haveSamples = true;
		} else if (a == "--depths" && i + 1 < argc) depthsPath = argv[++i];
		else if (a == "--sam" && i + 1 < argc) samDir = argv[++i];
		else if (a == "--mismatches" && i + 1 < argc) {
			char *end = NULL;
			const long d = strtol(argv[++i], &end, 10);
			if (!*argv[i] || *end || d < 0 || d > OGB_MAP_MAX_MISMATCHES) {
				cerr << "ogb_overlap: --mismatches takes 0 to " << OGB_MAP_MAX_MISMATCHES << ", not " << argv[i] << endl;
				return 1;
			}
			maxMismatches = (int)d;
		} else {
			cerr << "Usage: ogb_overlap -l minOverlap [-pe n files...] [-se n files...] [-f prefix] [-s] [--dump file] [--resave file] [--unitigs file] [--coverage file] [--samples n files... --depths file [--mismatches d] [--sam dir]]" << endl;
			return a == "-h" || a == "--help" ? 0 : 1;
		}
	}
	if (minimumOverlapLength == 0 || (pairedEndFileNames.empty() && singleEndFileNames.empty())) {
		cerr << "ogb_overlap: need -l and at least one input file" << endl;
		return 1;
	}
	if (startFromUnitigGraph && unitigsPath) {
		cerr << "ogb_overlap: --unitigs needs the build on the device; -s resumes from a .unitig file without one" << endl;
		return 1;
	}
	if (startFromUnitigGraph && coveragePath) {
		cerr << "ogb_overlap: --coverage needs the build on the device; -s resumes from a .unitig file without one" << endl;
		return 1;
	}
	if (haveSamples != (depthsPath != NULL) || (haveSamples && sampleFileNames.empty())) {
		cerr << "ogb_overlap: --samples (at least one file) and --depths go together" << endl;
		return 1;
	}
	if (maxMismatches >= 0 && (!haveSamples || startFromUnitigGraph)) {
		cerr << "ogb_overlap: --mismatches needs --samples and --depths, on the build on the device (not with -s)" << endl;
		return 1;
	}
	if (samDir) {
		set<string> seen;
		bool clash = false;
		for (size_t j = 0; j < sampleFileNames.size(); j++) {
			const size_t slash = sampleFileNames[j].find_last_of('/');
			clash |= !seen.insert(slash == string::npos ? sampleFileNames[j] : sampleFileNames[j].substr(slash + 1)).second;
		}
		if (!haveSamples || !depthsPath || startFromUnitigGraph || clash) {
			cerr << "ogb_overlap: --sam needs --samples and --depths, on the build on the device (not with -s), and samples of distinct basenames" << endl;
			return 1;
		}
	}
	if (startFromUnitigGraph && depthsPath) {
		cerr << "ogb_overlap: --samples / --depths need the build on the device; -s resumes from a .unitig file without one" << endl;
		return 1;
	}
	try {
		Dataset *dataSet = new Dataset(pairedEndFileNames, singleEndFileNames, minimumOverlapLength);	// main.cpp:33
		OverlapGraph *overlapGraph;
		if (startFromUnitigGraph) {																		// main.cpp:36-42: no GPU involved
			overlapGraph = new OverlapGraph();
			overlapGraph->setDataset(dataSet);
			overlapGraph->readGraphFromFile(allFileName + ".unitig");
			overlapGraph->sortEdges();
			if (dumpPath) dumpGraph(dumpPath, dataSet, overlapGraph, minimumOverlapLength);
			if (resavePath) overlapGraph->saveGraphToFile(resavePath);
			cout << "reads: " << dataSet->getNumberOfReads() << " unique: " << dataSet->getNumberOfUniqueReads()
			     << " nodes: " << overlapGraph->getNumberOfNodes() << " edges: " << overlapGraph->getNumberOfEdges() << " (from " << allFileName << ".unitig)" << endl;
			delete dataSet;
			delete overlapGraph;
			return 0;
		}
		if (dumpPath) OverlapGraph::simplifyInBuild = false;											// --dump wants the graph as it is at OverlapGraph.cpp:210
		if (unitigsPath || coveragePath || depthsPath) OverlapGraph::spellInBuild = true;
		HashTable *hashTable = new HashTable();															// main.cpp:45
		hashTable->insertDataset(dataSet, minimumOverlapLength);										// main.cpp:46
		overlapGraph = new OverlapGraph(hashTable); //hashTable deleted by this function after building the graph (main.cpp:47)
		if (allFileName != "") dataSet->saveReads(allFileName + "_sortedReads.fasta");					// main.cpp:48
		if (dumpPath) {
			dumpGraph(dumpPath, dataSet, overlapGraph, minimumOverlapLength);
			overlapGraph->simplifyGraph();																// ... and then the rest of the constructor (:211-215)
		}
		if (matesPath) dumpMates(matesPath, dataSet);
		overlapGraph->sortEdges();																		// main.cpp:49
		if (allFileName != "") overlapGraph->saveGraphToFile(allFileName + ".unitig");					// main.cpp:50
		const ogb_stats &st = overlapGraph->getBuildStats();
		const ogb_simplify_stats &ss = overlapGraph->getSimplifyStats();
		cout << "reads: " << dataSet->getNumberOfReads() << " unique: " << dataSet->getNumberOfUniqueReads()
		     << " nodes: " << overlapGraph->getNumberOfNodes() << " edges: " << overlapGraph->getNumberOfEdges()
		     << " device ms: " << st.ms_total << " + simplification " << ss.ms << " (" << ss.merges << " merges, " << ss.dead_ends << " dead ends, "
		     << ss.iterations << " iterations, " << ss.rounds << " rounds)" << endl;
		if (coveragePath) {
			overlapGraph->saveUnitigCoverageToFile(coveragePath);
			const ogb_coverage_stats &cv = overlapGraph->getCoverageStats();
			cout << "coverage: " << cv.unitigs << " unitigs " << cv.bases << " bases " << cv.placements << " placements " << cv.contained_placements
			     << " contained placements " << cv.unplaced << " unplaced, coverage device ms: " << cv.ms << " (" << coveragePath << ")" << endl;
		}
		if (depthsPath) {
			if (samDir && mkdir(samDir, 0777) != 0 && errno != EEXIST) throw OgbFailure(OGB_E_IO, string("cannot create ") + samDir);
			overlapGraph->saveSampleDepthsToFile(depthsPath, sampleFileNames, maxMismatches > 0 ? (uint32_t)maxMismatches : 0, samDir ? samDir : "");
			for (size_t j = 0; j < sampleFileNames.size(); j++) {
				const ogb_map_stats &mp = overlapGraph->getMapStats()[j];
				const size_t slash = sampleFileNames[j].find_last_of('/');
				cout << "map: " << (slash == string::npos ? sampleFileNames[j] : sampleFileNames[j].substr(slash + 1)) << " reads " << mp.reads_in
				     << " filtered " << mp.filtered << " mapped " << mp.mapped << " multi " << mp.multi << " placements " << mp.placements
				     << ", map device ms: " << mp.ms << " (" << depthsPath << ")" << endl;
			}
		}
		if (unitigsPath) {
			overlapGraph->saveUnitigsToFile(unitigsPath);
			const ogb_spell_stats &sp = overlapGraph->getSpellStats();
			cout << "unitigs: " << sp.unitigs << " bases: " << sp.bases << " spell device ms: " << sp.ms << " (" << unitigsPath << ")" << endl;
		}
		delete dataSet;
		delete overlapGraph;
	} catch (const OgbFailure &e) {
		cerr << "ogb_overlap: " << e.what() << endl;
		return 2;
	}
	return 0;
}
