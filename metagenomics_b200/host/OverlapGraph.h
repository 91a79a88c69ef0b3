// OverlapGraph.h -- drop-in for the graph-construction half of MetaGenomics/OverlapGraph.h:32-76.
//
// OverlapGraph(HashTable*) runs the reference's buildOverlapGraphFromHashTable (OverlapGraph.cpp:
// 107-215) on the GPU -- contained-read marking, window scan with exact verification, transitive
// reduction, and the closing fix-point of contractCompositePaths + removeDeadEndNodes (:211-215) --
// and leaves the state the reference has when the function returns: graph[1..N] of linked twin Edge
// objects with their composite read lists, numberOfNodes / numberOfEdges, Read::superReadID, mate-pair
// lists filled after containment marking, hash table freed. With OverlapGraph::simplifyInBuild = false
// the build stops at `delete hashTable` (:210, the graph before the fix-point) and keeps the table's
// device context until simplifyGraph() is called. The host stages that follow in the reference
// (calculateFlow and the simplification loops of main.cpp) consume that state unchanged and are not
// part of this library.
//
// The per-read member functions of the reference build (checkOverlap, insertAllEdgesOfRead,
// markTransitiveEdges, ...) are kept with their signatures and semantics as host code over the same
// data, so code written against the reference header keeps compiling; the constructor does not call
// them.
#ifndef OGB_HOST_OVERLAPGRAPH_H_
#define OGB_HOST_OVERLAPGRAPH_H_

#include "Common.h"
#include "Dataset.h"
#include "Edge.h"
#include "HashTable.h"

enum nodeType { UNEXPLORED = 0, EXPLORED = 1, EXPLORED_AND_TRANSITIVE_EDGES_MARKED = 2 };
enum markType { VACANT = 0, INPLAY = 1, ELIMINATED = 2 };

class OverlapGraph
{
	private:
		Dataset *dataSet;
		HashTable *hashTable;
		vector<vector<Edge *> *> *graph;
		UINT64 numberOfNodes;
		UINT64 numberOfEdges;
		UINT64 hashStringLength;						// kept after the table is freed (checkOverlap needs it)
		ogb_stats lastStats;
		UINT8 twinEdgeOrientation(UINT8 orientation);
		void materialise(const ogb_edge *edges, UINT64 n);
		void clearGraph(void);
		ogb_simplify_stats lastSimplifyStats;
		ogb_spell_stats lastSpellStats;
		ogb_coverage_stats lastCoverageStats;
		vector<ogb_map_stats> lastMapStats;

	public:
		bool flowComputed;
		static bool simplifyInBuild;					// true (default): the build ends with the fix-point of :211-215, like the reference's
		static bool spellInBuild;						// false (default); true: simplifyGraph() also spells the canonical unitigs on the device
														// (getStringInEdge, :2009) and keeps the hash table's device context for saveUnitigsToFile
		OverlapGraph(void);
		OverlapGraph(HashTable *ht);
		~OverlapGraph();
		bool buildOverlapGraphFromHashTable(HashTable *ht);
		bool simplifyGraph(void);						// :211-215 on the device (only after a build with simplifyInBuild == false); frees the hash table
		void markContainedReads(void);
		bool checkOverlap(Read *read1, Read *read2, UINT64 orient, UINT64 start);
		bool checkOverlapForContainedRead(Read *read1, Read *read2, UINT64 orient, UINT64 start);
		bool insertAllEdgesOfRead(UINT64 readNumber, vector<nodeType> *exploredReads);
		bool markTransitiveEdges(UINT64 readNumber, vector<markType> *markedNodes);
		bool removeTransitiveEdges(UINT64 readNumber);
		bool insertEdge(Edge *edge);
		bool insertEdge(Read *read1, Read *read2, UINT8 orient, UINT16 overlapOffset);
		UINT64 getNumberOfEdges(void) { return numberOfEdges; }
		UINT64 getNumberOfNodes(void) { return numberOfNodes; }
		bool setDataset(Dataset *dataset) { dataSet = dataset; dataset->readMatePairsFromFile(); return true; }
		void sortEdges();
		bool saveGraphToFile(string fileName);			// OverlapGraph.cpp:1219-1259: the reference's .unitig text format
		bool saveUnitigCoverageToFile(string fileName);	// per-base read depth of the spelled unitigs as TSV (ogb_graph_coverage); before saveUnitigsToFile
		bool saveSampleDepthsToFile(string fileName, const vector<string> &sampleFiles);	// every sample file mapped onto the spelled unitigs
														// (ogb_graph_map_reads), the depth table in MetaBAT's layout (ogb_graph_write_depths); before saveUnitigsToFile
		bool saveUnitigsToFile(string fileName);		// the unitigs spelled in the build as FASTA (ogb_graph_write_unitigs); frees the hash table
		bool readGraphFromFile(string fileName);		// OverlapGraph.cpp:1267-1367 (resume path, main.cpp:36-42)
		Edge *findEdge(UINT64 source, UINT64 destination);
		bool isEdgePresent(UINT64 source, UINT64 destination);
		vector<vector<Edge *> *> *getGraph(void) { return graph; }
		const ogb_stats &getBuildStats(void) const { return lastStats; }
		const ogb_simplify_stats &getSimplifyStats(void) const { return lastSimplifyStats; }
		const ogb_spell_stats &getSpellStats(void) const { return lastSpellStats; }
		const ogb_coverage_stats &getCoverageStats(void) const { return lastCoverageStats; }
		const vector<ogb_map_stats> &getMapStats(void) const { return lastMapStats; }	// one per sample of saveSampleDepthsToFile
};

#endif
