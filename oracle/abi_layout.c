/* TEST INFRASTRUCTURE.  Prints the layout of channel_t / msgblk_t and the constants the reference's API
 * fixes, from the header named by -DHDR: built against the reference's acarsdec.h as _ref/abi_layout
 * (oracle/Makefile) and against include/acarsdec_compat.h by tests/test_compat.py, which compares the two. */
#include <stdio.h>
#include <stddef.h>
#include HDR
#define P(t, f) printf(#t "." #f " %zu\n", offsetof(t, f))
int main(void) {
  printf("sizeof(channel_t) %zu\nsizeof(msgblk_t) %zu\n", sizeof(channel_t), sizeof(msgblk_t));
  P(channel_t, chn); P(channel_t, Fr); P(channel_t, wf); P(channel_t, dm_buffer); P(channel_t, MskPhi); P(channel_t, MskDf);
  P(channel_t, MskClk); P(channel_t, MskLvlSum); P(channel_t, MskBitCount); P(channel_t, MskS); P(channel_t, idx);
  P(channel_t, inb); P(channel_t, outbits); P(channel_t, nbits); P(channel_t, Acarsstate); P(channel_t, blk); P(channel_t, th);
  P(msgblk_t, prev); P(msgblk_t, chn); P(msgblk_t, tv); P(msgblk_t, len); P(msgblk_t, err); P(msgblk_t, lvl); P(msgblk_t, txt); P(msgblk_t, crc);
  printf("MAXNBCHANNELS %d INTRATE %d WSYN %d END %d\n", MAXNBCHANNELS, INTRATE, (int)WSYN, (int)END);
  return 0; }
