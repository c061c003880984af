// tests/opening_book_host.cpp -- TEST SCAFFOLDING: compiles subproc_b200/csrc/opening_book.cuh for the host so the
// tree the playout kernel walks can be compared with the oracle without a GPU.
#include <string.h>
#include "../subproc_b200/csrc/opening_book.cuh"

static std::vector<obb::BookNode> g_nodes;

// builds the tree to `depth` plies; its node count, or -1 when build_book refuses (a node above the last ply without
// a legal move)
extern "C" long ob_book_build(int depth)
{
    return obb::build_book(depth, g_nodes) ? (long)g_nodes.size() : -1;
}

// the nodes of the last successful build, 32 bytes each
extern "C" void ob_book_copy(void *out)
{
    memcpy(out, g_nodes.data(), g_nodes.size() * sizeof(obb::BookNode));
}
