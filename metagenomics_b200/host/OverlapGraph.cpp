// OverlapGraph.cpp -- see OverlapGraph.h.
#include "OverlapGraph.h"

#include <cstdlib>
#include <cstring>

static bool byDestination(Edge *a, Edge *b) { return a->getDestinationRead()->getReadNumber() < b->getDestinationRead()->getReadNumber(); }
static bool byOffset(Edge *a, Edge *b) { return a->getOverlapOffset() < b->getOverlapOffset(); }

bool OverlapGraph::simplifyInBuild = true;
bool OverlapGraph::spellInBuild = false;

OverlapGraph::OverlapGraph(void)
	: dataSet(NULL), hashTable(NULL), graph(new vector<vector<Edge *> *>), numberOfNodes(0), numberOfEdges(0), hashStringLength(0), flowComputed(false)
{
	memset(&lastStats, 0, sizeof lastStats);
	memset(&lastSimplifyStats, 0, sizeof lastSimplifyStats);
	memset(&lastSpellStats, 0, sizeof lastSpellStats);
	memset(&lastCoverageStats, 0, sizeof lastCoverageStats);
}

OverlapGraph::OverlapGraph(HashTable *ht)
	: dataSet(NULL), hashTable(NULL), graph(new vector<vector<Edge *> *>), numberOfNodes(0), numberOfEdges(0), hashStringLength(0), flowComputed(false)
{
	memset(&lastStats, 0, sizeof lastStats);
	memset(&lastSimplifyStats, 0, sizeof lastSimplifyStats);
	memset(&lastSpellStats, 0, sizeof lastSpellStats);
	memset(&lastCoverageStats, 0, sizeof lastCoverageStats);
	buildOverlapGraphFromHashTable(ht);
}

void OverlapGraph::clearGraph(void)
{
	for (size_t i = 0; i < graph->size(); i++) {
		for (size_t j = 0; j < graph->at(i)->size(); j++) delete graph->at(i)->at(j);
		delete graph->at(i);
	}
	graph->clear();
	numberOfNodes = numberOfEdges = 0;
}

OverlapGraph::~OverlapGraph()
{
	clearGraph();
	delete graph;
	delete hashTable;														// only still there after a build that stopped at :210
}

// OverlapGraph.cpp:841-855
UINT8 OverlapGraph::twinEdgeOrientation(UINT8 orientation)
{
	static const UINT8 twin[4] = {3, 1, 2, 0};
	if (orientation > 3) throw OgbFailure(OGB_E_ARG, "Unsupported edge orientation.");
	return twin[orientation];
}

// OverlapGraph.cpp:107-210 on the device.
bool OverlapGraph::buildOverlapGraphFromHashTable(HashTable *ht)
{
	flowComputed = false;
	if (hashTable != ht) delete hashTable;									// a table left over from a build that stopped at :210
	hashTable = ht;
	dataSet = ht->getDataset();
	hashStringLength = ht->getHashStringLength();
	clearGraph();
	graph->reserve(dataSet->getNumberOfUniqueReads() + 1);
	for (UINT64 i = 0; i <= dataSet->getNumberOfUniqueReads(); i++) graph->push_back(new vector<Edge *>);	// :131-138

	markContainedReads();													// :140
	if (getenv("OGB_MATES_ON_HOST") == NULL) dataSet->setMatePairContext(ht->getContext());	// batched lookup on the GPU (ogb_mate_lookup)
	dataSet->readMatePairsFromFile();										// :142 (needs superReadID)
	dataSet->setMatePairContext(NULL);

	ogb_context *ctx = ht->getContext();
	ogbCheck(ogb_build_graph(ctx, 0), "OverlapGraph::buildOverlapGraphFromHashTable");	// :144-204
	ogbCheck(ogb_get_stats(ctx, &lastStats), "OverlapGraph");
	if (simplifyInBuild) return simplifyGraph();							// :211-215; the graph at :210 never leaves the device
	uint64_t n = 0;
	ogbCheck(ogb_graph_edge_count(ctx, 0, &n), "OverlapGraph");
	void *pinned = NULL;
	ogbCheck(ogb_alloc_host(&pinned, (n ? n : 1) * sizeof(ogb_edge)), "OverlapGraph");
	int rc = ogb_graph_edges(ctx, 0, (ogb_edge *)pinned, n);
	if (rc == OGB_OK) materialise((const ogb_edge *)pinned, n);
	ogb_free_host(pinned);
	ogbCheck(rc, "OverlapGraph");
	return true;															// the table (and its device context) stays until simplifyGraph() or the destructor
}

// OverlapGraph.cpp:211-215 on the device: do { contractCompositePaths(); removeDeadEndNodes(); } while (counter > 0), then the
// Edge objects of the simplified graph -- composite edges with their three lists (Edge.h:30-32), linked to their reverse edges.
bool OverlapGraph::simplifyGraph(void)
{
	if (!hashTable) throw OgbFailure(OGB_E_STATE, "simplifyGraph: the hash table (and its device context) has been freed");
	ogb_context *ctx = hashTable->getContext();
	ogbCheck(ogb_graph_simplify(ctx, &lastSimplifyStats), "OverlapGraph::simplifyGraph");
	const uint64_t ne = lastSimplifyStats.n_edges_out, ni = lastSimplifyStats.n_items;
	vector<ogb_cedge> edges(ne ? ne : 1);
	vector<ogb_clist_item> items(ni ? ni : 1);
	ogbCheck(ogb_graph_composite_edges(ctx, edges.data(), ne, items.data(), ni), "OverlapGraph::simplifyGraph");
	const UINT64 nodes = graph->size();
	clearGraph();
	for (UINT64 i = 0; i < nodes; i++) graph->push_back(new vector<Edge *>);
	vector<Edge *> objs(ne, (Edge *)NULL);
	for (uint64_t e = 0; e < ne; e++) {
		const ogb_cedge &x = edges[e];
		vector<UINT64> *listReads = new vector<UINT64>(x.count);
		vector<UINT16> *listOverlapOffsets = new vector<UINT16>(x.count);
		vector<UINT8> *listOrientations = new vector<UINT8>(x.count);
		for (uint32_t k = 0; k < x.count; k++) {
			const ogb_clist_item &it = items[x.list_start + k];
			listReads->at(k) = it.read; listOverlapOffsets->at(k) = it.offset; listOrientations->at(k) = it.orient;
		}
		objs[e] = new Edge(dataSet->getReadFromID(x.src), dataSet->getReadFromID(x.dst), x.orient, x.offset, listReads, listOverlapOffsets, listOrientations);
		insertEdge(objs[e]);
	}
	for (uint64_t e = 0; e < ne; e++) objs[e]->setReverseEdge(objs[edges[e].twin]);
	if (spellInBuild) {														// the sequences of the canonical unitigs (getStringInEdge, :2009)
		ogbCheck(ogb_graph_spell(ctx, 1, 0, UINT64_MAX, &lastSpellStats), "OverlapGraph::simplifyGraph");
		return true;														// they stay on the device, with the table, until saveUnitigsToFile
	}
	delete hashTable;														// :210 -- the graph owns and frees the table
	hashTable = NULL;
	return true;
}

// Per-base read depth of the unitigs simplifyGraph() spelled (spellInBuild), weighted by the Dataset's read frequencies and with the
// contained reads placed in their super reads, written as TSV (ogb_graph_write_coverage). The device context stays: call it before
// saveUnitigsToFile, which releases it.
bool OverlapGraph::saveUnitigCoverageToFile(string fileName)
{
	if (!hashTable) throw OgbFailure(OGB_E_STATE, "saveUnitigCoverageToFile: no unitigs on the device (set OverlapGraph::spellInBuild before the build)");
	ogb_context *ctx = hashTable->getContext();
	const uint64_t n = dataSet->getNumberOfUniqueReads();
	ogbCheck(ogb_graph_coverage(ctx, ogb_dataset_frequencies(dataSet->handle()), n, &lastCoverageStats), "OverlapGraph::saveUnitigCoverageToFile");
	ogbCheck(ogb_graph_write_coverage(ctx, fileName.c_str()), "OverlapGraph::saveUnitigCoverageToFile");
	return true;
}

// Maps the reads of every sample file (FASTA or FASTQ, read by the Dataset's parser) onto the unitigs simplifyGraph() spelled
// (spellInBuild), with up to maxMismatches substitutions per read (0: exact occurrences only), and writes their depths as one table in MetaBAT's layout, one column pair per sample named after the file's basename
// (ogb_graph_write_depths). The device context stays: call it before saveUnitigsToFile, which releases it.
bool OverlapGraph::saveSampleDepthsToFile(string fileName, const vector<string> &sampleFiles, uint32_t maxMismatches)
{
	if (!hashTable) throw OgbFailure(OGB_E_STATE, "saveSampleDepthsToFile: no unitigs on the device (set OverlapGraph::spellInBuild before the build)");
	ogb_context *ctx = hashTable->getContext();
	lastMapStats.assign(sampleFiles.size(), ogb_map_stats());
	vector<string> names(sampleFiles.size());
	vector<const char *> cnames(sampleFiles.size());
	for (size_t j = 0; j < sampleFiles.size(); j++) {
		ogb_dataset *ds = NULL;
		ogbCheck(ogb_dataset_create(&ds), "OverlapGraph::saveSampleDepthsToFile");
		const char *bases = NULL;
		const uint64_t *offsets = NULL;
		uint64_t n = 0;
		int rc = ogb_dataset_add_file(ds, sampleFiles[j].c_str());
		if (rc == OGB_OK) rc = ogb_dataset_raw_reads(ds, &bases, &offsets, &n);
		if (rc == OGB_OK) rc = ogb_graph_map_reads_approx(ctx, bases, offsets, n, maxMismatches, NULL, NULL, &lastMapStats[j]);
		ogb_dataset_destroy(ds);
		ogbCheck(rc, "OverlapGraph::saveSampleDepthsToFile");
		const size_t slash = sampleFiles[j].find_last_of('/');
		names[j] = slash == string::npos ? sampleFiles[j] : sampleFiles[j].substr(slash + 1);
		cnames[j] = names[j].c_str();
	}
	ogbCheck(ogb_graph_write_depths(ctx, fileName.c_str(), cnames.data()), "OverlapGraph::saveSampleDepthsToFile");
	return true;
}

// The unitigs simplifyGraph() spelled (spellInBuild) as FASTA, decoded on the device; then the table and its context go, as at :210.
bool OverlapGraph::saveUnitigsToFile(string fileName)
{
	if (!hashTable) throw OgbFailure(OGB_E_STATE, "saveUnitigsToFile: no unitigs on the device (set OverlapGraph::spellInBuild before the build)");
	ogbCheck(ogb_graph_write_unitigs(hashTable->getContext(), fileName.c_str()), "OverlapGraph::saveUnitigsToFile");
	delete hashTable;
	hashTable = NULL;
	return true;
}

// Builds the linked Edge objects from the flat, canonically sorted edge list. The twin of
// (u,v,o,off) is (v,u,twin(o),(UINT16)(L_v+off-L_u)) (OverlapGraph.cpp:410-412); identical tuples
// (reverse-complement self-overlaps are held twice) pair up with each other.
void OverlapGraph::materialise(const ogb_edge *edges, UINT64 n)
{
	vector<Edge *> objs(n, (Edge *)NULL);
	vector<UINT64> first(dataSet->getNumberOfUniqueReads() + 2, 0);
	for (UINT64 e = 0; e < n; e++) first[edges[e].src + 1]++;
	for (size_t i = 1; i < first.size(); i++) first[i] += first[i - 1];		// edges of node u: [first[u], first[u+1])
	for (UINT64 e = 0; e < n; e++) {
		objs[e] = new Edge(dataSet->getReadFromID(edges[e].src), dataSet->getReadFromID(edges[e].dst), edges[e].orient, edges[e].offset);
		insertEdge(objs[e]);
	}
	for (UINT64 e = 0; e < n; e++) {
		if (objs[e]->getReverseEdge() != NULL) continue;
		const ogb_edge &x = edges[e];
		UINT16 want_off = (UINT16)(dataSet->getReadFromID(x.dst)->getReadLength() + x.offset - dataSet->getReadFromID(x.src)->getReadLength());
		UINT8 want_o = twinEdgeOrientation(x.orient);
		for (UINT64 t = first[x.dst]; t < first[x.dst + 1]; t++) {
			if (t == e || objs[t]->getReverseEdge() != NULL) continue;
			if (edges[t].dst == x.src && edges[t].orient == want_o && edges[t].offset == want_off) {
				objs[e]->setReverseEdge(objs[t]);
				objs[t]->setReverseEdge(objs[e]);
				break;
			}
		}
		if (objs[e]->getReverseEdge() == NULL) throw OgbFailure(OGB_E_STATE, "edge without twin");
	}
}

// OverlapGraph.cpp:225-290 on the device; copies Read::superReadID back.
void OverlapGraph::markContainedReads(void)
{
	ogb_context *ctx = hashTable->getContext();
	ogbCheck(ogb_mark_contained(ctx), "OverlapGraph::markContainedReads");
	UINT64 n = dataSet->getNumberOfUniqueReads();
	vector<uint64_t> sup(n + 1, 0);
	ogbCheck(ogb_super_read_ids(ctx, sup.data(), n + 1), "OverlapGraph::markContainedReads");
	for (UINT64 i = 1; i <= n; i++) dataSet->getReadFromID(i)->superReadID = sup[i];
}

// OverlapGraph.cpp:390-400
bool OverlapGraph::insertEdge(Edge *edge)
{
	UINT64 id = edge->getSourceRead()->getReadNumber();
	if (graph->at(id)->empty()) numberOfNodes++;
	graph->at(id)->push_back(edge);
	numberOfEdges++;
	return true;
}

// OverlapGraph.cpp:407-419
bool OverlapGraph::insertEdge(Read *read1, Read *read2, UINT8 orient, UINT16 overlapOffset)
{
	Edge *forward = new Edge(read1, read2, orient, overlapOffset);
	UINT16 back = (UINT16)(read2->getReadLength() + overlapOffset - read1->getReadLength());
	Edge *reverse = new Edge(read2, read1, twinEdgeOrientation(orient), back);
	forward->setReverseEdge(reverse);
	reverse->setReverseEdge(forward);
	insertEdge(forward);
	insertEdge(reverse);
	return true;
}

// OverlapGraph.cpp:354-383 (host strings; the device restates it on packed words in K3)
bool OverlapGraph::checkOverlap(Read *read1, Read *read2, UINT64 orient, UINT64 start)
{
	string s1 = read1->getStringForward();
	string s2 = (orient < 2) ? read2->getStringForward() : read2->getStringReverse();
	UINT64 h = hashStringLength;
	if ((orient & 1) == 0) {
		if (s1.size() - start - h >= s2.size() - h) return false;
		UINT64 n = s1.size() - (start + h);
		return s1.compare(start + h, n, s2, h, n) == 0;
	}
	if (s2.size() - h < start) return false;
	return s1.compare(0, start, s2, s2.size() - h - start, start) == 0;
}

// OverlapGraph.cpp:302-340
bool OverlapGraph::checkOverlapForContainedRead(Read *read1, Read *read2, UINT64 orient, UINT64 start)
{
	string s1 = read1->getStringForward();
	string s2 = (orient < 2) ? read2->getStringForward() : read2->getStringReverse();
	UINT64 h = hashStringLength;
	UINT64 rest2 = s2.size() - h;
	if ((orient & 1) == 0) {
		UINT64 rest1 = s1.size() - start - h;
		return rest1 >= rest2 && s1.compare(start + h, rest2, s2, h, rest2) == 0;
	}
	return start >= rest2 && s1.compare(start - rest2, rest2, s2, 0, rest2) == 0;
}

// OverlapGraph.cpp:529-565 (needs a live hash table, i.e. only usable before the build frees it)
bool OverlapGraph::insertAllEdgesOfRead(UINT64 readNumber, vector<nodeType> *exploredReads)
{
	if (!hashTable) throw OgbFailure(OGB_E_STATE, "insertAllEdgesOfRead: the hash table has been freed");
	Read *read1 = dataSet->getReadFromID(readNumber);
	string text = read1->getStringForward();
	UINT64 h = hashTable->getHashStringLength();
	for (UINT64 j = 1; j < read1->getReadLength() - h; j++) {
		vector<UINT64> *hits = hashTable->getListOfReads(text.substr(j, h));
		for (size_t k = 0; k < hits->size(); k++) {
			UINT64 data = hits->at(k), o = data >> 62;
			Read *read2 = dataSet->getReadFromID(data & 0X3FFFFFFFFFFFFFFF);
			if (exploredReads->at(read2->getReadNumber()) != UNEXPLORED) continue;
			if (read1->superReadID != 0 || read2->superReadID != 0 || !checkOverlap(read1, read2, o, j)) continue;
			UINT16 overlap = (o & 1) ? (UINT16)(h + j) : (UINT16)(read1->getReadLength() - j);
			static const UINT8 orientationOf[4] = {3, 0, 2, 1};
			insertEdge(read1, read2, orientationOf[o], (UINT16)(read1->getReadLength() - overlap));
		}
	}
	if (!graph->at(readNumber)->empty()) sort(graph->at(readNumber)->begin(), graph->at(readNumber)->end(), byOffset);
	return true;
}

// OverlapGraph.cpp:574-615
bool OverlapGraph::markTransitiveEdges(UINT64 readNumber, vector<markType> *markedNodes)
{
	vector<Edge *> *mine = graph->at(readNumber);
	for (size_t i = 0; i < mine->size(); i++) markedNodes->at(mine->at(i)->getDestinationRead()->getReadNumber()) = INPLAY;
	for (size_t i = 0; i < mine->size(); i++) {
		UINT64 pivot = mine->at(i)->getDestinationRead()->getReadNumber();
		if (markedNodes->at(pivot) != INPLAY) continue;
		UINT8 t1 = mine->at(i)->getOrientation();
		vector<Edge *> *theirs = graph->at(pivot);
		for (size_t j = 0; j < theirs->size(); j++) {
			UINT64 w = theirs->at(j)->getDestinationRead()->getReadNumber();
			UINT8 t2 = theirs->at(j)->getOrientation();
			if (markedNodes->at(w) == INPLAY && (t1 & 1) == ((t2 >> 1) & 1)) markedNodes->at(w) = ELIMINATED;
		}
	}
	for (size_t i = 0; i < mine->size(); i++)
		if (markedNodes->at(mine->at(i)->getDestinationRead()->getReadNumber()) == ELIMINATED) {
			mine->at(i)->transitiveRemovalFlag = true;
			mine->at(i)->getReverseEdge()->transitiveRemovalFlag = true;
		}
	for (size_t i = 0; i < mine->size(); i++) markedNodes->at(mine->at(i)->getDestinationRead()->getReadNumber()) = VACANT;
	markedNodes->at(readNumber) = VACANT;
	return true;
}

// OverlapGraph.cpp:623-661
bool OverlapGraph::removeTransitiveEdges(UINT64 readNumber)
{
	vector<Edge *> *mine = graph->at(readNumber);
	for (size_t i = 0; i < mine->size(); i++) {
		if (!mine->at(i)->transitiveRemovalFlag) continue;
		Edge *twin = mine->at(i)->getReverseEdge();
		vector<Edge *> *theirs = graph->at(twin->getSourceRead()->getReadNumber());
		for (size_t k = 0; k < theirs->size(); k++)
			if (theirs->at(k) == twin) {
				delete twin;
				theirs->at(k) = theirs->back();
				theirs->pop_back();
				if (theirs->empty()) numberOfNodes--;
				numberOfEdges--;
				break;
			}
	}
	size_t kept = 0;
	for (size_t i = 0; i < mine->size(); i++) {
		if (!mine->at(i)->transitiveRemovalFlag) mine->at(kept++) = mine->at(i);
		else { numberOfEdges--; delete mine->at(i); }
	}
	mine->resize(kept);
	if (mine->empty()) numberOfNodes--;
	return true;
}

// OverlapGraph.cpp:2799-2808
void OverlapGraph::sortEdges()
{
	for (UINT64 i = 1; i < graph->size(); i++)
		if (!graph->at(i)->empty()) sort(graph->at(i)->begin(), graph->at(i)->end(), byDestination);
}

Edge *OverlapGraph::findEdge(UINT64 source, UINT64 destination)
{
	for (size_t i = 0; i < graph->at(source)->size(); i++)
		if (graph->at(source)->at(i)->getDestinationRead()->getReadNumber() == destination) return graph->at(source)->at(i);
	throw OgbFailure(OGB_E_ARG, "Cannot find edge");
}

bool OverlapGraph::isEdgePresent(UINT64 source, UINT64 destination)
{
	for (size_t i = 0; i < graph->at(source)->size(); i++)
		if (graph->at(source)->at(i)->getDestinationRead()->getReadNumber() == destination) return true;
	return false;
}

// OverlapGraph.cpp:1219-1259 -- the reference's .unitig format: one decimal number per line; for every edge with
// source < destination (a self-edge: one of the twin pair), source, destination, orientation, overlapOffset, the number
// of reads inside the edge and, for each of them, read number, overlap offset, orientation. The reference picks the
// self-edge twin with the lower heap address; here it is the one that sits first in the node's list (the same edge for a
// graph that came out of readGraphFromFile, where the forward edge is created and inserted first).
bool OverlapGraph::saveGraphToFile(string fileName)
{
	FILE *f = fopen(fileName.c_str(), "w");
	if (!f) throw OgbFailure(OGB_E_IO, "Unable to open file: " + fileName);
	for (UINT64 i = 1; i < graph->size(); i++) {
		vector<Edge *> *l = graph->at(i);
		for (UINT64 j = 0; j < l->size(); j++) {
			Edge *e = l->at(j);
			const UINT64 source = e->getSourceRead()->getReadNumber(), destination = e->getDestinationRead()->getReadNumber();
			bool write = source < destination;
			if (source == destination) {											// the twin is in the same list: keep the first of the two
				write = true;
				for (UINT64 k = 0; k < j; k++) if (l->at(k) == e->getReverseEdge()) { write = false; break; }
			}
			if (!write) continue;
			fprintf(f, "%llu\n%llu\n%llu\n%llu\n%llu\n", (unsigned long long)source, (unsigned long long)destination, (unsigned long long)e->getOrientation(),
			        (unsigned long long)e->getOverlapOffset(), (unsigned long long)e->getListOfReads()->size());
			for (UINT64 k = 0; k < e->getListOfReads()->size(); k++)
				fprintf(f, "%llu\n%llu\n%llu\n", (unsigned long long)e->getListOfReads()->at(k), (unsigned long long)e->getListOfOverlapOffsets()->at(k),
				        (unsigned long long)e->getListOfOrientations()->at(k));
		}
	}
	if (fclose(f) != 0) throw OgbFailure(OGB_E_IO, "Unable to write file: " + fileName);
	return true;
}

// OverlapGraph.cpp:1267-1367 -- rebuilds the graph (every edge together with its reverse edge, whose read list, offsets and
// orientations are derived as in :1321-1341) from a .unitig file; the Dataset must be the one the file was written for.
bool OverlapGraph::readGraphFromFile(string fileName)
{
	FILE *f = fopen(fileName.c_str(), "r");
	if (!f) throw OgbFailure(OGB_E_IO, "Unable to open file: " + fileName);
	vector<UINT64> list;
	unsigned long long t;
	while (fscanf(f, "%llu", &t) == 1) list.push_back(t);
	fclose(f);
	for (size_t i = 0; i < graph->size(); i++) {
		for (size_t j = 0; j < graph->at(i)->size(); j++) delete graph->at(i)->at(j);
		delete graph->at(i);
	}
	graph->clear();
	numberOfNodes = numberOfEdges = 0;
	for (UINT64 i = 0; i <= dataSet->getNumberOfUniqueReads(); i++) graph->push_back(new vector<Edge *>);
	for (size_t i = 0; i + 5 <= list.size();) {
		const UINT64 source = list[i++], destination = list[i++], orientation = list[i++], overlapOffset = list[i++], nReads = list[i++];
		if (i + 3 * nReads > list.size()) throw OgbFailure(OGB_E_IO, "Truncated unitig file: " + fileName);
		vector<UINT64> *listReads = new vector<UINT64>;
		vector<UINT16> *listOverlapOffsets = new vector<UINT16>;
		vector<UINT8> *listOrientations = new vector<UINT8>;
		UINT64 length = 0;
		for (UINT64 j = 0; j < 3 * nReads; j += 3) {
			listReads->push_back(list[i + j]);
			listOverlapOffsets->push_back((UINT16)list[i + j + 1]);
			listOrientations->push_back((UINT8)list[i + j + 2]);
			length += list[i + j + 1];
		}
		Read *read1 = dataSet->getReadFromID(source), *read2 = dataSet->getReadFromID(destination);
		vector<UINT64> *listReadsReverse = new vector<UINT64>;
		vector<UINT16> *listOverlapOffsetsReverse = new vector<UINT16>;
		vector<UINT8> *listOrientationsReverse = new vector<UINT8>;
		const UINT64 size = listReads->size();
		for (UINT64 j = 0; j < size; j++) {											// :1321-1341
			listReadsReverse->push_back(listReads->at(size - j - 1));
			UINT64 length1, overlapOffsetForward;
			if (j == 0) { length1 = read2->getReadLength(); overlapOffsetForward = overlapOffset - length; }
			else { length1 = dataSet->getReadFromID(listReads->at(size - j))->getReadLength(); overlapOffsetForward = listOverlapOffsets->at(size - j); }
			const UINT64 length2 = dataSet->getReadFromID(listReads->at(size - j - 1))->getReadLength();
			listOverlapOffsetsReverse->push_back((UINT16)(length1 + overlapOffsetForward - length2));
			listOrientationsReverse->push_back(!(listOrientations->at(size - j - 1)));
		}
		const UINT64 reverseOverlapOffset = overlapOffset + read2->getReadLength() - read1->getReadLength();
		Edge *edgeForward = new Edge(), *edgeReverse = new Edge();
		edgeForward->makeEdge(read1, read2, orientation, overlapOffset, listReads, listOverlapOffsets, listOrientations);
		edgeReverse->makeEdge(read2, read1, twinEdgeOrientation((UINT8)orientation), reverseOverlapOffset, listReadsReverse, listOverlapOffsetsReverse, listOrientationsReverse);
		edgeForward->setReverseEdge(edgeReverse);
		edgeReverse->setReverseEdge(edgeForward);
		insertEdge(edgeForward);
		insertEdge(edgeReverse);
		i += nReads * 3;
	}
	return true;
}
