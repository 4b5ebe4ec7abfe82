package sw ;

import java.nio.charset.StandardCharsets ;
import java.util.List ;

/**
 * JNI binding of libswb200 for the reference's own runtime (Java 1.8 / Spark 1.5.2, pom.xml:17-32):
 * {@code System.loadLibrary("swbjni")} loads jni/swb_jni.c, which forwards every method below to the
 * C ABI of include/swb200.h.  Handles are opaque {@code long}s; sequences cross as Latin-1 bytes plus
 * {@code long[] offsets} (n + 1 entries); a native failure surfaces as an unchecked RuntimeException
 * carrying swb_last_error(), because Function3.call declares no checked exception
 * (reference SmithWaterman.java:62).
 *
 * NOT COMPILED OR RUN in the build environment (no JDK there).  tests/test_abi_and_host.py checks that
 * every {@code static native} method below has a {@code Java_sw_NativeSW_*} export with the same argument
 * count in the compiled shim.  A Panama FFM (JDK 22+) binding of the same ABI is under java/ffm/.
 */
final class NativeSW
{
	static { System.loadLibrary( System.getProperty( "swb.jni" , "swbjni" ) ) ; }

	private NativeSW() {}

	// ---- context ------------------------------------------------------------------------
	static native String lastError() ;
	static native int deviceCount() ;
	static native long create( int device , long workspaceBytes ) ;
	static native void destroy( long ctx ) ;

	// ---- reference set (HBM-resident, 2-bit packed) ----------------------------------------
	static native long refsetLoad( long ctx , byte[] bytes , long[] offsets ) ;
	static native void refsetFree( long refset ) ;

	// ---- align all reads x all references of the set --------------------------------------
	static native long align( long ctx , long refset , byte[] readBytes , long[] readOffsets , int match , int mismatch , int gap , int flags ) ;
	/** one pair through the native submission queue (swb_align_pair): concurrent calls are coalesced into one launch sequence */
	static native long alignPair( long ctx , byte[] ref , byte[] read , int match , int mismatch , int gap , int flags ) ;
	/** hits mode (swb_align_hits): every pair scored, only each read's topK best pairs with score >= minScore traced */
	static native long alignHits( long ctx , long refset , byte[] readBytes , long[] readOffsets , int match , int mismatch , int gap , int flags , int topK , int minScore ) ;
	static native void resultFree( long result ) ;

	// ---- result arrays ---------------------------------------------------------------------
	static native int[] scores( long result ) ;
	static native int[] refTotals( long result ) ;
	static native int[] bestHits( long result ) ;
	/** hits mode: {score, ref, i, j} x topK per read, padding (0, -1, 0, 0); empty for a plain result */
	static native int[] resultHits( long result ) ;
	/** all-hits mode (swb_align_all_hits): every pair with score >= minScore and >= the read's best score - margin traced */
	static native long alignAllHits( long ctx , long refset , byte[] readBytes , long[] readOffsets , int match , int mismatch , int gap , int flags , int minScore , int margin ) ;
	/** all-hits mode: nReads + 1 offsets into resultHitList; empty for any other result */
	static native long[] resultHitOffsets( long result ) ;
	/** all-hits mode: {score, ref, i, j} per listed pair, read by read, score descending then ref ascending */
	static native int[] resultHitList( long result ) ;
	static native long[] cellOffsets( long result ) ;
	static native int[] cells( long result ) ;
	static native int[] beginnings( long result ) ;
	static native int[] opLens( long result ) ;
	static native long pairCellCount( long result , long pair ) ;
	static native int[] pairCell( long result , long pair , long k ) ;
	static native byte[][] materialize( long result , long cell , int opLen , byte[] ref , byte[] read ) ;

	// ---- multi-GPU (one JVM, several devices) -----------------------------------------------
	static native long multiCreate( int[] devices , long workspaceBytes ) ;
	static native void multiDestroy( long multi ) ;
	static native void multiRefsetLoad( long multi , byte[] bytes , long[] offsets ) ;
	static native long[] multiShardRefs( long multi , int shard ) ;
	static native long multiAlign( long multi , byte[] readBytes , long[] readOffsets , int match , int mismatch , int gap , int flags ) ;
	static native long multiAlignHits( long multi , byte[] readBytes , long[] readOffsets , int match , int mismatch , int gap , int flags , int topK , int minScore ) ;
	static native long multiShard( long multiResult , int shard ) ;
	static native int[] multiBestHits( long multiResult , int nReads ) ;
	static native int[] multiResultHits( long multiResult , int nReads ) ;
	static native void multiResultFree( long multiResult ) ;

	static final int F_SCORES_ONLY = 1 , F_NO_FETCH = 2 , F_TIE_GT = 4 ;
	/** every read and its reverse complement: results over 2 * nRefs oriented references, o = 2r + strand (swb200.h) */
	static final int F_BOTH_STRANDS = 8 ;

	/** process-wide engine context on CUDA device -Dswb.device (default 0); thread-safe on the native side */
	private static long ctx = 0 ;
	static synchronized long context()
	{
		if( ctx == 0 )
		{
			ctx = create( Integer.getInteger( "swb.device" , 0 ).intValue() , Long.getLong( "swb.workspace" , 0L ).longValue() ) ;
			Runtime.getRuntime().addShutdownHook( new Thread() { public void run() { destroy( ctx ) ; } } ) ;
		}
		return ctx ;
	}

	/** sequences -> concatenated Latin-1 bytes; offsets[k] .. offsets[k+1] delimit sequence k */
	static byte[] pack( List<String> seqs , long[] offsets )
	{
		long total = 0 ;
		for( int k = 0 ; k < seqs.size() ; k++ ) { offsets[k] = total ; total += seqs.get(k).length() ; }
		offsets[seqs.size()] = total ;
		if( total > Integer.MAX_VALUE - 8 ) throw new RuntimeException( "sequence batch exceeds a Java array: split the call" ) ;
		byte[] bytes = new byte[(int) total] ;
		for( int k = 0 ; k < seqs.size() ; k++ )
		{
			byte[] b = seqs.get(k).getBytes( StandardCharsets.ISO_8859_1 ) ;
			System.arraycopy( b , 0 , bytes , (int) offsets[k] , b.length ) ;
		}
		return bytes ;
	}
}
