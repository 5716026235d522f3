// Host build of the thread-per-read exact routing with classify_runs' rotation memo counted (tools/memo_hits.py).
#define ET_MEMO_STATS
#include "../tests/native/exact_thread_check.cpp"

extern "C" long etc_memo_runs() { return trew::et::memo_runs; }
extern "C" long etc_memo_hits() { return trew::et::memo_hits; }
extern "C" void etc_memo_reset() { trew::et::memo_runs = trew::et::memo_hits = 0; }
