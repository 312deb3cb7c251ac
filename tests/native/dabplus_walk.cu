// Host driver of superframe_walk (dabplus.cuh) as the DAB+ pass runs it: walk, decode what the walk attempts without an
// outcome (here: take the outcome from stdin), repeat until a walk lists nothing new.
// stdin: lines "n_frames" then n_frames - 4 pre_ok flags, then n_frames - 4 ok flags (windows of fewer than 5 frames: none).
// stdout per stream: "<rounds> <decoded> <attempted windows...>"
#include "dabplus.cuh"

#include <cstdio>
#include <vector>

int main()
{
  int n;
  while (scanf("%d", &n) == 1)
  {
    const int nw = n >= 5 ? n - 4 : 0;
    std::vector<int> pre(nw), ok(nw);
    for (int & v : pre) if (scanf("%d", &v) != 1) return 1;
    for (int & v : ok) if (scanf("%d", &v) != 1) return 1;
    std::vector<uint8_t> state(nw + 1);
    for (int w = 0; w < nw; w++) state[w] = pre[w] ? dab::SF_PRE_OK : 0;
    std::vector<int> att(nw + 1);
    int rounds = 0, decoded = 0, n_att = 0;
    while (true)
    {
      n_att = dab::superframe_walk(state.data(), n, att.data());
      rounds++;
      int fresh = 0;
      for (int k = 0; k < n_att; k++)
        if (!(state[att[k]] & dab::SF_DECODED)) { state[att[k]] |= dab::SF_DECODED | (ok[att[k]] ? dab::SF_OK : 0); fresh++; }
      if (fresh == 0) break;
      decoded += fresh;
    }
    printf("%d %d", rounds, decoded);
    for (int k = 0; k < n_att; k++) printf(" %d", att[k]);
    printf("\n");
  }
  return 0;
}
